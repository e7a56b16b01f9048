"""ctypes binding of include/b200probe.h.

The product path has NO fallback: if libb200probe.so is missing this module raises on import of
the library handle, and every probe call raises ProbeError when CUDA is unavailable.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200PROBE_LIB") or os.path.join(_HERE, "libb200probe.so")     # B200PROBE_LIB: another build of the SAME library (kernel experiments); there is still no fallback

ABI_VERSION = 2
MAX_DEVICES = 64
IPC_HANDLE_BYTES = 64

HBM_READ, HBM_WRITE, HBM_COPY = 1, 2, 4
VARIANT_TMA, VARIANT_DIRECT = 0, 1
A2A_PEER_ALL, A2A_PEER_PAIR, A2A_NCCL, A2A_CE = 0, 1, 2, 3
PAIR_SHARE, PAIR_ISOLATED, PAIR_STEPPED = 0, 1, 2
GEMM_EXACT, GEMM_UNIFORM = 0, 1
GEMM_FILL_E4M3 = 4          # b200probe_gemm_fill / _operand_bits: bit 2 of `which` selects E4M3 operands (one byte per element)
MEMTEST_VERIFY, MEMTEST_WRITE = 1, 2
A2A_AUTO, A2A_PULL_TMA, A2A_PUSH_TMA, A2A_PUSH_DIRECT, A2A_PUSH_BUF, A2A_MIX_TMA, A2A_PUSH_STAGGER, A2A_PUSH_SYNC = 0, 1, 2, 3, 4, 5, 6, 7
A2A_SYNC_BYTES = 4096
NVML_ERROR_TIMEOUT = 10
EVENT_XID_CRITICAL = 0x8
EVENT_DBE = 0x2
EVENT_SBE = 0x1


class Device(C.Structure):
    _fields_ = [
        ("index", C.c_int),
        ("uuid", C.c_char * 96),
        ("name", C.c_char * 96),
        ("pci_bus_id", C.c_char * 32),
        ("mem_total", C.c_uint64),
        ("cc_major", C.c_int),
        ("cc_minor", C.c_int),
        ("numa_node", C.c_int),
        ("mig_enabled", C.c_int),
        ("supported_events", C.c_uint64),
        ("cuda_ordinal", C.c_int),
    ]


class HealthEvent(C.Structure):
    _fields_ = [
        ("rc_wait", C.c_int),
        ("event_type", C.c_uint64),
        ("event_data", C.c_uint64),
        ("gpu_instance_id", C.c_uint32),
        ("compute_instance_id", C.c_uint32),
        ("device_index", C.c_int),
        ("skipped", C.c_int),
        ("newly_unhealthy", C.c_uint64),
    ]


class NvlinkStatus(C.Structure):
    _fields_ = [
        ("links_total", C.c_int),
        ("links_active", C.c_int),
        ("active_mask", C.c_uint32),
        ("fabric_state", C.c_int),
        ("fabric_status", C.c_int),
        ("fabric_health_mask", C.c_uint32),
        ("data_tx_kib", C.c_uint64),
        ("data_rx_kib", C.c_uint64),
        ("raw_tx_kib", C.c_uint64),
        ("raw_rx_kib", C.c_uint64),
        ("counters_ok", C.c_int),
    ]


class Busy(C.Structure):
    _fields_ = [
        ("compute_procs", C.c_int),
        ("util_gpu_pct", C.c_int),
        ("util_mem_pct", C.c_int),
        ("mem_used", C.c_uint64),
        ("busy", C.c_int),
    ]


class HbmCfg(C.Structure):
    _fields_ = [
        ("min_bytes", C.c_uint64),
        ("max_bytes", C.c_uint64),
        ("modes", C.c_int),
        ("warmup", C.c_int),
        ("reps", C.c_int),
        ("seed", C.c_uint32),
        ("variant", C.c_int),
        ("verify", C.c_int),
        ("flush_l2", C.c_int),
        ("stage_bytes", C.c_int),
        ("stages", C.c_int),
        ("warps_per_cta", C.c_int),
        ("ctas_per_sm", C.c_int),
        ("launches_per_rep", C.c_int),
    ]


class HbmResult(C.Structure):
    _fields_ = [
        ("bytes", C.c_uint64),
        ("mode", C.c_int),
        ("variant", C.c_int),
        ("ms_median", C.c_double),
        ("ms_best", C.c_double),
        ("gbs_median", C.c_double),
        ("gbs_best", C.c_double),
        ("sum64", C.c_uint64),
        ("xor32", C.c_uint32),
        ("verified", C.c_int),
        ("cache_resident", C.c_int),
    ]


class A2aCfg(C.Structure):
    _fields_ = [
        ("bytes_per_pair", C.c_uint64),
        ("mode", C.c_int),
        ("warmup", C.c_int),
        ("reps", C.c_int),
        ("seed", C.c_uint32),
        ("verify", C.c_int),
        ("ctas_per_peer", C.c_int),
        ("variant", C.c_int),
    ]


class A2aResult(C.Structure):
    _fields_ = [
        ("g", C.c_int),
        ("ms_median", C.c_double),
        ("ms_best", C.c_double),
        ("egress_gbs", C.c_double * MAX_DEVICES),
        ("ingress_gbs", C.c_double * MAX_DEVICES),
        ("min_pair_gbs", C.c_double),
        ("max_pair_gbs", C.c_double),
        ("verified", C.c_int),
        ("pair_source", C.c_int),
    ]


class GemmCfg(C.Structure):
    _fields_ = [
        ("m", C.c_int),
        ("n", C.c_int),
        ("k", C.c_int),
        ("warmup", C.c_int),
        ("reps", C.c_int),
        ("seed", C.c_uint32),
        ("samples", C.c_int),
        ("operands", C.c_int),
        ("sustain_seconds", C.c_double),
    ]


class GemmResult(C.Structure):
    _fields_ = [
        ("m", C.c_int),
        ("n", C.c_int),
        ("k", C.c_int),
        ("ms_median", C.c_double),
        ("ms_best", C.c_double),
        ("tflops_median", C.c_double),
        ("tflops_best", C.c_double),
        ("tflops_sustained", C.c_double),
        ("max_abs_err", C.c_double),
        ("max_rel_err", C.c_double),
        ("samples", C.c_int),
        ("bad", C.c_int),
        ("c_sum64", C.c_uint64),
        ("c_xor32", C.c_uint32),
        ("verified", C.c_int),
        ("operands", C.c_int),
        ("max_err_over_tol", C.c_double),
    ]


class EccStatus(C.Structure):
    _fields_ = [
        ("ecc_mode", C.c_int),
        ("corrected_volatile", C.c_int64),
        ("uncorrected_volatile", C.c_int64),
        ("remap_corrected_rows", C.c_int),
        ("remap_uncorrected_rows", C.c_int),
        ("remap_pending", C.c_int),
        ("remap_failure", C.c_int),
    ]


class MemtestCfg(C.Structure):
    _fields_ = [
        ("fraction", C.c_double),
        ("max_bytes", C.c_uint64),
        ("min_bytes", C.c_uint64),
        ("chunk_bytes", C.c_uint64),
        ("passes", C.c_int),
        ("seed", C.c_uint32),
    ]


class MemtestResult(C.Structure):
    _fields_ = [
        ("bytes_tested", C.c_uint64),
        ("chunks", C.c_int),
        ("passes", C.c_int),
        ("free_before", C.c_uint64),
        ("total", C.c_uint64),
        ("alloc_ms", C.c_double),
        ("test_ms", C.c_double),
        ("gbs", C.c_double),
        ("bad_words", C.c_uint64),
        ("first_bad_word", C.c_uint64),
        ("bad_bits", C.c_uint32),
        ("first_bad_element", C.c_int),
        ("ecc_corrected_delta", C.c_int64),
        ("ecc_uncorrected_delta", C.c_int64),
        ("ecc_after", EccStatus),
    ]


_P = C.POINTER
_vp = C.c_void_p

# name -> (restype, argtypes); the single source of truth for "every symbol include/*.h declares"
SIGNATURES = {
    "b200probe_abi_version": (C.c_int, []),
    "b200probe_init": (C.c_int, [C.c_char_p]),
    "b200probe_shutdown": (None, []),
    "b200probe_strerror": (C.c_char_p, [C.c_int]),
    "b200probe_last_error": (C.c_int, [C.c_char_p, C.c_int]),
    "b200probe_device_count": (C.c_int, [_P(C.c_int)]),
    "b200probe_device_info": (C.c_int, [C.c_int, _P(Device)]),
    "b200probe_enumerate": (C.c_int, [_P(Device), C.c_int, _P(C.c_int), _P(C.c_double)]),
    "b200probe_health_open": (C.c_int, [C.c_char_p, _P(C.c_uint64)]),
    "b200probe_health_wait": (C.c_int, [C.c_int, _P(HealthEvent)]),
    "b200probe_passive_health": (C.c_int, [C.c_int, _P(C.c_uint64)]),
    "b200probe_health_mask": (C.c_int, [_P(C.c_uint64)]),
    "b200probe_health_close": (None, []),
    "b200probe_device_busy": (C.c_int, [C.c_int, _P(Busy)]),
    "b200probe_nvlink_passive": (C.c_int, [C.c_int, _P(NvlinkStatus)]),
    "b200probe_hbm_sweep": (C.c_int, [C.c_int, _P(HbmCfg), _P(HbmResult), C.c_int, _P(C.c_int)]),
    "b200probe_hbm_release": (C.c_int, [C.c_int]),
    "b200probe_hbm_fill": (C.c_int, [C.c_int, _vp, C.c_uint64, C.c_uint32, _P(HbmCfg), _vp]),
    "b200probe_hbm_copy": (C.c_int, [C.c_int, _vp, _vp, C.c_uint64, _P(HbmCfg), _vp]),
    "b200probe_hbm_read": (C.c_int, [C.c_int, _vp, C.c_uint64, _vp, _P(HbmCfg), _vp]),
    "b200probe_hbm_copy_host": (C.c_int, [C.c_int, _vp, _vp, C.c_uint64, _P(C.c_uint64), _P(C.c_uint32)]),
    "b200probe_hbm_verify": (C.c_int, [C.c_int, _vp, C.c_uint64, C.c_uint32, _P(C.c_uint64), _P(C.c_uint32), _P(C.c_uint64), _P(C.c_uint64)]),
    "b200probe_hbm_ecc": (C.c_int, [C.c_int, _P(EccStatus)]),
    "b200probe_memtest_element": (C.c_int, [C.c_int, _vp, C.c_uint64, C.c_uint64, C.c_int, C.c_uint32, C.c_uint32, _P(C.c_uint64), _P(C.c_uint64),
                                            _P(C.c_uint32)]),
    "b200probe_hbm_memtest": (C.c_int, [C.c_int, _P(MemtestCfg), _P(MemtestResult)]),
    "b200probe_host_alloc": (C.c_int, [C.c_uint64, _P(_vp)]),
    "b200probe_host_free": (C.c_int, [_vp]),
    "b200probe_nvlink_a2a": (C.c_int, [_P(C.c_int), C.c_int, _P(A2aCfg), _P(C.c_double), _P(A2aResult)]),
    "b200probe_a2a_release": (C.c_int, []),
    "b200probe_enable_peer_access": (C.c_int, [_P(C.c_int), C.c_int]),
    "b200probe_a2a_window_create": (C.c_int, [C.c_int, C.c_int, C.c_uint64, _P(_vp), C.c_char_p]),
    "b200probe_a2a_window_import": (C.c_int, [C.c_int, C.c_char_p, _P(_vp)]),
    "b200probe_a2a_window_release": (C.c_int, [C.c_int, _vp, C.c_int]),
    "b200probe_a2a_window_fill": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_uint64, C.c_uint32, _vp]),
    "b200probe_a2a_exchange": (C.c_int, [C.c_int, C.c_int, C.c_int, _P(_vp), C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, _vp]),
    "b200probe_a2a_chunk_seed": (C.c_uint32, [C.c_uint32, C.c_int, C.c_int]),
    "b200probe_gemm": (C.c_int, [C.c_int, _P(GemmCfg), _P(GemmResult)]),
    "b200probe_gemm_release": (C.c_int, [C.c_int]),
    "b200probe_gemm_operand_bits": (C.c_uint16, [C.c_uint64, C.c_uint32, C.c_int]),
    "b200probe_gemm_launch": (C.c_int, [C.c_int, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "b200probe_gemm_fill": (C.c_int, [C.c_int, _vp, C.c_uint64, C.c_uint32, C.c_int, _vp]),
    "b200probe_gemm_fp8": (C.c_int, [C.c_int, _P(GemmCfg), _P(GemmResult)]),
    "b200probe_gemm_fp8_launch": (C.c_int, [C.c_int, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "b200probe_pattern_word": (C.c_uint32, [C.c_uint64, C.c_uint32]),
}

_lib = None


def load() -> C.CDLL:
    """Load libb200probe.so and declare every signature.  Raises (never falls back) when missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C k3s-nvidia_b200/csrc`. There is no CPU/PyTorch fallback for the probe path."
        )
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_LOCAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError = ABI drift; let it propagate
        fn.restype = res
        fn.argtypes = args
    if lib.b200probe_abi_version() != ABI_VERSION:
        raise ImportError(f"libb200probe.so ABI {lib.b200probe_abi_version()} != {ABI_VERSION}")
    _lib = lib
    return lib
