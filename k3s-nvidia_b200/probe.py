"""Python face of the C ABI (include/b200probe.h).  Thin: every method is one C call.

The reference stack has no code for this path (SURVEY.md §0); the calls mirror what the plugin
installed by /root/reference/README.md:116 does with NVML (enumerate, XID event wait) and add the
active probes (HBM sweep, NVLink all-to-all, tcgen05 GEMM).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

from . import _lib as L

MODE_NAME = {L.HBM_READ: "read", L.HBM_WRITE: "write", L.HBM_COPY: "copy"}


class ProbeError(RuntimeError):
    def __init__(self, rc: int, what: str, detail: str):
        self.rc = rc
        super().__init__(f"{what}: rc={rc} ({detail})")


@dataclass
class DeviceInfo:
    index: int
    uuid: str
    name: str
    pci_bus_id: str
    mem_total: int
    cc: tuple
    numa_node: int
    mig_enabled: int
    supported_events: int
    cuda_ordinal: int


@dataclass
class HbmPoint:
    bytes: int
    mode: str
    variant: int
    ms_median: float
    ms_best: float
    gbs_median: float
    gbs_best: float
    sum64: int
    xor32: int
    verified: int
    cache_resident: bool


@dataclass
class A2aReport:
    g: int
    ms_median: float
    ms_best: float
    egress_gbs: List[float]
    ingress_gbs: List[float]
    pair_gbs: List[List[float]]
    min_pair_gbs: float
    max_pair_gbs: float
    verified: int
    pair_source: int = 0       # _lib.PAIR_SHARE / PAIR_ISOLATED / PAIR_STEPPED


@dataclass
class GemmReport:
    m: int
    n: int
    k: int
    ms_median: float
    ms_best: float
    tflops_median: float
    tflops_best: float
    tflops_sustained: float
    max_abs_err: float
    max_rel_err: float
    samples: int
    bad: int
    c_sum64: int
    c_xor32: int
    verified: int
    operands: int = 0            # _lib.GEMM_EXACT / GEMM_UNIFORM
    max_err_over_tol: float = 0.0


@dataclass
class MemtestReport:
    """b200probe_memtest_result_t; ECC and remap fields are -1 where NVML cannot report them."""
    bytes_tested: int
    chunks: int
    passes: int
    free_before: int
    total: int
    alloc_ms: float
    test_ms: float
    gbs: float
    bad_words: int
    first_bad_word: int
    bad_bits: int
    first_bad_element: int
    ecc_corrected_delta: int
    ecc_uncorrected_delta: int
    remap_corrected_rows: int
    remap_uncorrected_rows: int
    remap_pending: int
    remap_failure: int


@dataclass
class HealthEvent:
    rc_wait: int
    event_type: int
    event_data: int
    device_index: int
    skipped: bool
    newly_unhealthy: int
    timed_out: bool = field(default=False)


def _hbm_cfg(**kw) -> L.HbmCfg:
    cfg = L.HbmCfg()
    for k, v in kw.items():
        if v is not None:
            setattr(cfg, k, v)
    return cfg


class Probe:
    """One process-wide handle on libb200probe.so."""

    def __init__(self, nvml_path: Optional[str] = None):
        self.lib = L.load()
        self._check(self.lib.b200probe_init(nvml_path.encode() if nvml_path else None), "b200probe_init")

    # -- plumbing ------------------------------------------------------------------------------
    def _check(self, rc: int, what: str) -> None:
        if rc != 0:
            buf = C.create_string_buffer(512)
            self.lib.b200probe_last_error(buf, 512)
            detail = buf.value.decode(errors="replace") or self.lib.b200probe_strerror(rc).decode()
            raise ProbeError(rc, what, detail)

    def close(self) -> None:
        self.lib.b200probe_shutdown()

    # -- enumeration ---------------------------------------------------------------------------
    def device_count(self) -> int:
        n = C.c_int()
        self._check(self.lib.b200probe_device_count(C.byref(n)), "device_count")
        return n.value

    @staticmethod
    def _dev(d: L.Device) -> DeviceInfo:
        return DeviceInfo(d.index, d.uuid.decode(), d.name.decode(), d.pci_bus_id.decode(), d.mem_total,
                          (d.cc_major, d.cc_minor), d.numa_node, d.mig_enabled, d.supported_events, d.cuda_ordinal)

    def device_info(self, idx: int) -> DeviceInfo:
        d = L.Device()
        self._check(self.lib.b200probe_device_info(idx, C.byref(d)), "device_info")
        return self._dev(d)

    def enumerate(self):
        """Re-read the device list from NVML; returns (devices, microseconds)."""
        arr = (L.Device * L.MAX_DEVICES)()
        n = C.c_int()
        us = C.c_double()
        self._check(self.lib.b200probe_enumerate(arr, L.MAX_DEVICES, C.byref(n), C.byref(us)), "enumerate")
        return [self._dev(arr[i]) for i in range(n.value)], us.value

    # -- passive health ------------------------------------------------------------------------
    def health_open(self, disable_healthchecks: Optional[str] = None) -> int:
        m = C.c_uint64()
        arg = disable_healthchecks.encode() if disable_healthchecks is not None else None
        self._check(self.lib.b200probe_health_open(arg, C.byref(m)), "health_open")
        return m.value

    def health_wait(self, timeout_ms: int) -> HealthEvent:
        ev = L.HealthEvent()
        self._check(self.lib.b200probe_health_wait(timeout_ms, C.byref(ev)), "health_wait")
        return HealthEvent(ev.rc_wait, ev.event_type, ev.event_data, ev.device_index, bool(ev.skipped),
                           ev.newly_unhealthy, ev.rc_wait == L.NVML_ERROR_TIMEOUT)

    def passive_health(self, timeout_ms: int) -> int:
        m = C.c_uint64()
        self._check(self.lib.b200probe_passive_health(timeout_ms, C.byref(m)), "passive_health")
        return m.value

    def health_mask(self) -> int:
        m = C.c_uint64()
        self._check(self.lib.b200probe_health_mask(C.byref(m)), "health_mask")
        return m.value

    def health_close(self) -> None:
        self.lib.b200probe_health_close()

    # -- is somebody else on the device? ---------------------------------------------------------------
    def device_busy(self, idx: int) -> dict:
        b = L.Busy()
        self._check(self.lib.b200probe_device_busy(idx, C.byref(b)), "device_busy")
        return {f: getattr(b, f) for f, _ in L.Busy._fields_}

    # -- passive NVLink ------------------------------------------------------------------------------
    def nvlink_passive(self, idx: int) -> dict:
        st = L.NvlinkStatus()
        self._check(self.lib.b200probe_nvlink_passive(idx, C.byref(st)), "nvlink_passive")
        return {f: getattr(st, f) for f, _ in L.NvlinkStatus._fields_}

    # -- HBM -------------------------------------------------------------------------------------
    def hbm_sweep(self, idx: int = 0, *, min_bytes=None, max_bytes=None, modes=None, warmup=None, reps=None,
                  seed=None, variant=None, verify=1, flush_l2=None, stage_bytes=None, stages=None,
                  warps_per_cta=None, ctas_per_sm=None, launches_per_rep=None) -> List[HbmPoint]:
        cfg = _hbm_cfg(min_bytes=min_bytes, max_bytes=max_bytes, modes=modes, warmup=warmup, reps=reps, seed=seed,
                       variant=variant, verify=verify, flush_l2=flush_l2, stage_bytes=stage_bytes, stages=stages,
                       warps_per_cta=warps_per_cta, ctas_per_sm=ctas_per_sm, launches_per_rep=launches_per_rep)
        cap = 128
        out = (L.HbmResult * cap)()
        n = C.c_int()
        rc = self.lib.b200probe_hbm_sweep(idx, C.byref(cfg), out, cap, C.byref(n))
        pts = [HbmPoint(r.bytes, MODE_NAME[r.mode], r.variant, r.ms_median, r.ms_best, r.gbs_median, r.gbs_best,
                        r.sum64, r.xor32, r.verified, bool(r.cache_resident)) for r in out[: n.value]]
        self._check(rc, "hbm_sweep")
        return pts

    def hbm_fill(self, ordinal, dst_ptr, nbytes, seed, stream=0, **tuning):
        cfg = _hbm_cfg(**tuning) if tuning else None
        self._check(self.lib.b200probe_hbm_fill(ordinal, dst_ptr, nbytes, seed, C.byref(cfg) if cfg else None, stream), "hbm_fill")

    def hbm_copy(self, ordinal, src_ptr, dst_ptr, nbytes, stream=0, **tuning):
        cfg = _hbm_cfg(**tuning) if tuning else None
        self._check(self.lib.b200probe_hbm_copy(ordinal, src_ptr, dst_ptr, nbytes, C.byref(cfg) if cfg else None, stream), "hbm_copy")

    def hbm_read(self, ordinal, src_ptr, nbytes, partials_ptr, stream=0, **tuning):
        cfg = _hbm_cfg(**tuning) if tuning else None
        self._check(self.lib.b200probe_hbm_read(ordinal, src_ptr, nbytes, partials_ptr, C.byref(cfg) if cfg else None, stream), "hbm_read")

    def hbm_copy_host(self, ordinal: int, src, dst):
        """src, dst: writable buffers (numpy arrays / bytearrays) of equal size.  Returns (sum64, xor32)."""
        import numpy as np

        s = np.ascontiguousarray(src)
        d = dst
        assert d.flags["C_CONTIGUOUS"] and s.nbytes == d.nbytes
        s64, x32 = C.c_uint64(), C.c_uint32()
        self._check(self.lib.b200probe_hbm_copy_host(ordinal, s.ctypes.data, d.ctypes.data, s.nbytes, C.byref(s64), C.byref(x32)),
                    "hbm_copy_host")
        return s64.value, x32.value

    def hbm_verify(self, ordinal: int, ptr: int, nbytes: int, seed: int):
        """Verdict pass on a device buffer -> (sum64, xor32, bad_words, first_bad_word)."""
        s64, x32, bad, first = C.c_uint64(), C.c_uint32(), C.c_uint64(), C.c_uint64()
        self._check(self.lib.b200probe_hbm_verify(ordinal, ptr, nbytes, seed, C.byref(s64), C.byref(x32), C.byref(bad), C.byref(first)),
                    "hbm_verify")
        return s64.value, x32.value, bad.value, first.value

    # -- HBM integrity ---------------------------------------------------------------------------
    def memtest_element(self, ordinal: int, ptr: int, nbytes: int, base_word: int, flags: int, expect_seed: int, write_seed: int):
        """One march element on a device buffer -> (bad_words, first_bad_word, bad_bits)."""
        bad, first, bits = C.c_uint64(), C.c_uint64(), C.c_uint32()
        self._check(self.lib.b200probe_memtest_element(ordinal, ptr, nbytes, base_word, flags, expect_seed & 0xFFFFFFFF, write_seed & 0xFFFFFFFF,
                                                       C.byref(bad), C.byref(first), C.byref(bits)), "memtest_element")
        return bad.value, first.value, bits.value

    def hbm_ecc(self, idx: int) -> dict:
        st = L.EccStatus()
        self._check(self.lib.b200probe_hbm_ecc(idx, C.byref(st)), "hbm_ecc")
        return {f: getattr(st, f) for f, _ in L.EccStatus._fields_}

    def hbm_memtest(self, idx: int = 0, *, fraction=0.0, max_bytes=0, min_bytes=0, chunk_bytes=0, passes=0, seed=0) -> MemtestReport:
        cfg = L.MemtestCfg(fraction, max_bytes, min_bytes, chunk_bytes, passes, seed)
        r = L.MemtestResult()
        self._check(self.lib.b200probe_hbm_memtest(idx, C.byref(cfg), C.byref(r)), "hbm_memtest")
        e = r.ecc_after
        return MemtestReport(r.bytes_tested, r.chunks, r.passes, r.free_before, r.total, r.alloc_ms, r.test_ms, r.gbs, r.bad_words,
                             r.first_bad_word, r.bad_bits, r.first_bad_element, r.ecc_corrected_delta, r.ecc_uncorrected_delta,
                             e.remap_corrected_rows, e.remap_uncorrected_rows, e.remap_pending, e.remap_failure)

    def host_alloc(self, nbytes: int):
        """Pinned host buffer as a numpy uint8 array (free with host_free(arr))."""
        import numpy as np

        ptr = C.c_void_p()
        self._check(self.lib.b200probe_host_alloc(nbytes, C.byref(ptr)), "host_alloc")
        arr = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr.value))
        self._pinned = getattr(self, "_pinned", {})
        self._pinned[arr.ctypes.data] = ptr.value
        return arr

    def host_free(self, arr) -> None:
        ptr = getattr(self, "_pinned", {}).pop(arr.ctypes.data, None)
        if ptr is not None:
            self._check(self.lib.b200probe_host_free(ptr), "host_free")

    # -- NVLink ----------------------------------------------------------------------------------
    def nvlink_a2a(self, ordinals: Sequence[int], *, bytes_per_pair=None, mode=L.A2A_PEER_ALL, warmup=None, reps=None,
                   seed=0xB200, verify=1, ctas_per_peer=None, variant=L.A2A_AUTO) -> A2aReport:
        g = len(ordinals)
        cfg = L.A2aCfg()
        cfg.bytes_per_pair = bytes_per_pair or 0
        cfg.mode = mode
        cfg.warmup = warmup or 0
        cfg.reps = reps or 0
        cfg.seed = seed
        cfg.verify = verify
        cfg.ctas_per_peer = ctas_per_peer or 0
        cfg.variant = variant
        idx = (C.c_int * g)(*ordinals)
        pair = (C.c_double * (g * g))()
        res = L.A2aResult()
        rc = self.lib.b200probe_nvlink_a2a(idx, g, C.byref(cfg), pair, C.byref(res))
        self._check(rc, "nvlink_a2a")
        return A2aReport(g, res.ms_median, res.ms_best, list(res.egress_gbs[:g]), list(res.ingress_gbs[:g]),
                         [[pair[i * g + j] for j in range(g)] for i in range(g)], res.min_pair_gbs, res.max_pair_gbs,
                         res.verified, res.pair_source)

    def a2a_release(self) -> None:
        """Free the resident exchange context (windows, streams, NCCL communicators)."""
        self._check(self.lib.b200probe_a2a_release(), "a2a_release")

    # -- GEMM ------------------------------------------------------------------------------------
    def gemm(self, idx: int = 0, *, m=0, n=0, k=0, warmup=0, reps=0, seed=0xB200, samples=0, sustain_seconds=0.0, operands=L.GEMM_EXACT) -> GemmReport:
        cfg = L.GemmCfg(m, n, k, warmup, reps, seed, samples, operands, sustain_seconds)
        r = L.GemmResult()
        rc = self.lib.b200probe_gemm(idx, C.byref(cfg), C.byref(r))
        rep = GemmReport(r.m, r.n, r.k, r.ms_median, r.ms_best, r.tflops_median, r.tflops_best, r.tflops_sustained,
                         r.max_abs_err, r.max_rel_err, r.samples, r.bad, r.c_sum64, r.c_xor32, r.verified, r.operands, r.max_err_over_tol)
        self._check(rc, "gemm")
        return rep

    def gemm_fp8(self, idx: int = 0, *, m=0, n=0, k=0, warmup=0, reps=0, seed=0xB200, samples=0, sustain_seconds=0.0,
                 operands=L.GEMM_EXACT) -> GemmReport:
        """The FP8 tensor-core probe: E4M3 operands through tcgen05.mma kind::f8f6f4, bf16 C, with gemm()'s protocol and
        verdict rules.  m and n must be multiples of 256, k a multiple of 128."""
        cfg = L.GemmCfg(m, n, k, warmup, reps, seed, samples, operands, sustain_seconds)
        r = L.GemmResult()
        rc = self.lib.b200probe_gemm_fp8(idx, C.byref(cfg), C.byref(r))
        rep = GemmReport(r.m, r.n, r.k, r.ms_median, r.ms_best, r.tflops_median, r.tflops_best, r.tflops_sustained,
                         r.max_abs_err, r.max_rel_err, r.samples, r.bad, r.c_sum64, r.c_xor32, r.verified, r.operands, r.max_err_over_tol)
        self._check(rc, "gemm_fp8")
        return rep

    def gemm_fp8_launch(self, ordinal: int, a: int, b: int, c: int, m: int, n: int, k: int, stream=None) -> None:
        """One asynchronous E4M3 GEMM on device buffers: A [m][k], B [n][k] E4M3 row-major, C [m][n] bf16."""
        self._check(self.lib.b200probe_gemm_fp8_launch(ordinal, a, b, c, m, n, k, stream), "gemm_fp8_launch")

    def release(self, ordinals: Sequence[int] = ()) -> None:
        """Free every resident probe arena (HBM, GEMM per listed CUDA ordinal; the exchange context): what the plugin
        does after a probe round, so the daemon holds no device memory while tenants run."""
        for o in ordinals:
            self.lib.b200probe_hbm_release(o)
            self.lib.b200probe_gemm_release(o)
        self.lib.b200probe_a2a_release()
