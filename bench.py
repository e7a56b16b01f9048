#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the B200 health-probe path.

  python bench.py --gpus N --steps K --warmup W            (our arm; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  (the reference's CPU path, rank 0 only)

A step = one pass of the hot path over one batch of synthetic input = one HBM copy-probe launch
over a resident 1 GiB source (2 GiB algorithmic bytes: N read + N written), the size
BASELINE.json's configs[1] ("single-B200 HBM bandwidth probe, 1 MB-1 GB buffer sweep") takes its
verdict at.  value = aggregate GB/s over all ranks (weak scaling: one replica of the probe per
GPU, no data-path collective).  For N > 1 the NVLink all-to-all exchange (configs[2]) is measured
after the HBM region and reported under "nvlink".  See DESIGN.md §6 for every field.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries ONE JSON line: libraries that chat on fd 1 (NCCL prints its version banner there) are sent to
# stderr, and the result line goes to a private duplicate of the original stdout.
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit(line: dict) -> None:
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


GIB = 1 << 30
METRIC = "health-probe HBM GB/s & NVLink GB/s vs peak per GPU at 1/2/4/8 B200"
WORKLOAD = "configs[1]: single-B200 HBM bandwidth probe, copy pass at the 1 GiB verdict size of the 1 MiB-1 GiB sweep"
NVLINK_NOMINAL = 900.0
A2A_VARIANT = int(os.environ.get("B200PROBE_A2A_VARIANT", "0"))   # 0 AUTO (= PUSH_SYNC for the exchange), 1 PULL_TMA, 2 PUSH_TMA, 3 PUSH_DIRECT, 4 PUSH_BUF, 5 MIX_TMA, 6 PUSH_STAGGER, 7 PUSH_SYNC
NVLINK_GUIDE_ONE_WAY = 770.0   # /opt/skills/guides/B200_PROFILING.md: peer copy, ONE direction loaded; context only — the denominator
                               # used here is the two-way copy-engine exchange measured in the same run (nvlink.plugin_entry.copy_engines)


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    except (OSError, ValueError):
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


# ---- clock sampling during the timed region (NVML from a side thread; 10 ms period) --------------
class ClockSampler:
    def __init__(self, index: int):
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    _BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
             0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self._BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.01)

    def start(self):
        if self.nv:
            self.samples.clear()
            self._stop.clear()
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---- CPU legs (the only places bench.py may execute oracle/) -----------------------------------------
def load_oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle

    return _oracle, _oracle.load()


def cpu_copy_sample(o, threads: int, sample_bytes: int, target_s: float):
    """Time the oracle port of the copy pass on host memory: calibrate, then ~target_s of work.  Thread t is pinned to the
    t-th CPU of the process's allowed set, so a slice is first-touched and copied on one NUMA node every pass."""
    s, x = C.c_uint64(), C.c_uint32()
    t1 = o.oracle_host_sweep_pinned(sample_bytes, threads, 4, 2, 0xB200, C.byref(s), C.byref(x)) / 2
    reps = max(3, min(2000, int(target_s / max(t1, 1e-4))))
    dt = o.oracle_host_sweep_pinned(sample_bytes, threads, 4, reps, 0xB200, C.byref(s), C.byref(x))
    gbs = 2.0 * sample_bytes * reps / dt / 1e9
    return gbs, reps, dt, (s.value, x.value)


def nvml_poll_timing(o):
    """The reference's real path (passive NVML enumerate + XID event wait), timed on this host the way SURVEY.md
    §8d config 1 asks: 1000 iterations after 10 warm-ups, single thread; the C twin and, where importable, pynvml."""
    out = None
    try:
        if o.oracle_ph_open(None, None) != 0:
            return None
        allowed = os.sched_getaffinity(0)
        n_allowed = o.oracle_allowed_cpus()
        pinned_cpu = o.oracle_pin_self(0)                 # the single-thread figures are quoted pinned to one core
        o.oracle_ph_time_enumerate(10)
        o.oracle_ph_time_poll(10, 0)
        enum_us = o.oracle_ph_time_enumerate(1000)
        poll_us = o.oracle_ph_time_poll(1000, 0)
        out = {"enumerate_us": round(enum_us, 2), "poll_us": round(poll_us, 2), "polls_per_s": round(1e6 / max(poll_us, 1e-9)),
               "iters": 1000, "warmup": 10, "threads": 1, "pinned_to_cpu": pinned_cpu, "cpu_model": cpu_model(),
               "host_cpus": os.cpu_count(), "allowed_cpus": n_allowed}
        os.sched_setaffinity(0, allowed)                  # the N-thread variant and everything after run unpinned again
        # N-thread variant (SURVEY.md §8d config 1): one thread per GPU, each with its own event set on its device
        pps = C.c_double()
        n_gpus = len(_oracle_verdicts(o))
        us_n = o.oracle_ph_time_poll_threads(min(n_gpus, os.cpu_count() or 1), 1000, C.byref(pps))
        if us_n > 0:
            out["per_gpu_threads"] = {"threads": min(n_gpus, os.cpu_count() or 1), "poll_us": round(us_n, 2), "polls_per_s": round(pps.value)}
        o.oracle_ph_close()
    except Exception:  # noqa: BLE001
        return out
    try:
        import pynvml as nv

        nv.nvmlInit()

        def enumerate_once():
            for i in range(nv.nvmlDeviceGetCount()):
                h = nv.nvmlDeviceGetHandleByIndex(i)
                nv.nvmlDeviceGetUUID(h), nv.nvmlDeviceGetName(h), nv.nvmlDeviceGetMemoryInfo(h), nv.nvmlDeviceGetCudaComputeCapability(h)

        for _ in range(10):
            enumerate_once()
        t0 = time.perf_counter()
        for _ in range(1000):
            enumerate_once()
        out["pynvml_enumerate_us"] = round((time.perf_counter() - t0) * 1e3, 2)      # microseconds per enumerate (1000 iterations)
        nv.nvmlShutdown()
    except Exception:  # noqa: BLE001
        pass
    return out


def _oracle_verdicts(o):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle

    return _oracle.verdicts(o)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    _, o = load_oracle()
    cores = os.cpu_count() or 1
    sample_bytes = GIB
    s, x = C.c_uint64(), C.c_uint32()
    cores = o.oracle_allowed_cpus()
    sweep = o.oracle_host_sweep_pinned
    per = sweep(sample_bytes, cores, 4, 2, 0xB200, C.byref(s), C.byref(x)) / 2
    if per * (args.steps + args.warmup) > 150.0:
        sample_bytes = 256 << 20
        per = sweep(sample_bytes, cores, 4, 2, 0xB200, C.byref(s), C.byref(x)) / 2
    steps = args.steps
    if per * (steps + args.warmup) > 150.0:
        steps = max(1, int(150.0 / per) - args.warmup)
    if args.warmup:
        sweep(sample_bytes, cores, 4, args.warmup, 0xB200, C.byref(s), C.byref(x))
    dt = sweep(sample_bytes, cores, 4, steps, 0xB200, C.byref(s), C.byref(x))
    gbs = 2.0 * sample_bytes * steps / dt / 1e9
    sample = (f"copy pass over {sample_bytes >> 20} MiB of host memory per step, {steps} steps, {cores} pthreads each pinned to one CPU "
              f"({cpu_model()}; first touch and every pass of a slice on the same core) (oracle port; the reference ships no code)")
    line = {
        "impl": "reference", "metric": METRIC, "value": round(gbs, 2), "unit": "GB/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": round(dt / steps * 1e3, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "where": "host memory, CPU threads", "bytes_per_step": 2 * sample_bytes},
        "cpu_baseline": {"value": round(gbs, 2), "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(gbs, 2), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_path_nvml": nvml_poll_timing(o),
        "note": "the reference's own health path (passive NVML XID wait) moves 0 bytes; its timing is under reference_path_nvml",
    }
    emit(line)
    return 0


# ---- our arm -------------------------------------------------------------------------------------
def run_ours(args):
    import torch

    from k3s_nvidia_b200 import _lib as L
    from k3s_nvidia_b200 import dist as D
    from k3s_nvidia_b200.probe import Probe

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the probe path has no CPU fallback (use --impl reference for the CPU arm)")
    rank, local_rank, world = D.init()
    if world != args.gpus:
        raise SystemExit(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch N>1 with torchrun")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    p = Probe()
    nbytes = GIB
    seed = 0xB200
    src = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    p.hbm_fill(local_rank, src.data_ptr(), nbytes, seed, stream)
    torch.cuda.synchronize()

    nvml_index = local_rank          # NVML index of this rank's CUDA device (resolved by UUID inside the library)
    for i in range(p.device_count()):
        if p.device_info(i).cuda_ordinal == local_rank:
            nvml_index = i
    sampler = ClockSampler(nvml_index)

    def step():
        p.hbm_copy(local_rank, src.data_ptr(), dst.data_ptr(), nbytes, stream)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    D.barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    D.barrier()
    ms_local = e0.elapsed_time(e1)
    outputs = last_step_outputs(torch, p, local_rank, dst, stream) if args.dump_outputs and rank == 0 else None
    # sustained window next to the K-step figure (outside the timed region): back-to-back launches for >= 1 s, in batches of
    # 256 launches between two events; the clock sampler keeps running, so its summary covers a second of load
    sus_ms, sus_n = 0.0, 0
    while sus_ms < 1000.0:
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_.record()
        for _ in range(256):
            step()
        b_.record()
        b_.synchronize()
        sus_ms += a_.elapsed_time(b_)
        sus_n += 256
    sampler.stop()
    clocks = sampler.summary()             # taken NOW: the timed K steps + the >= 1 s sustained window, nothing else
    sustained = D.aggregate_bandwidth(2.0 * nbytes * sus_n, sus_ms)
    agg = D.aggregate_bandwidth(2.0 * nbytes * args.steps, ms_local)
    launch_ms = ms_local / args.steps

    # data result of the timed region (parity): dst == pattern, checked on the device + vs oracle on rank 0
    part = torch.zeros(4, dtype=torch.int64, device=dev)
    p.hbm_read(local_rank, dst.data_ptr(), nbytes, part.data_ptr(), stream)
    torch.cuda.synchronize()
    got = (part[0].item() & 0xFFFFFFFFFFFFFFFF, part[1].item() & 0xFFFFFFFF)

    # ---- e2e: the plugin-facing call, host cfg in -> host verdict out, every step -----------------
    e2e_steps = max(1, min(args.steps, 300))
    kw = dict(min_bytes=nbytes, max_bytes=nbytes, modes=L.HBM_COPY, warmup=0, reps=1, verify=1, seed=seed, launches_per_rep=1)   # one verdict = one copy
    for _ in range(min(3, max(1, args.warmup))):
        p.hbm_sweep(nvml_index, **kw)
    torch.cuda.synchronize()
    D.barrier()
    t0 = time.perf_counter()
    ok = True
    for _ in range(e2e_steps):
        pts = p.hbm_sweep(nvml_index, **kw)
        ok = ok and pts[0].verified == 1
    torch.cuda.synchronize()
    e2e_ms_local = (time.perf_counter() - t0) * 1e3
    D.barrier()
    e2e = D.aggregate_bandwidth(2.0 * nbytes * e2e_steps, e2e_ms_local)
    p.lib.b200probe_hbm_release(local_rank)

    # ---- NVLink all-to-all across ranks (the one exchange step), N > 1 -----------------------------
    nvlink = None
    if world > 1:
        nvlink = nvlink_exchange(torch, D, p, local_rank, rank, world, stream, args)
        # the code the DAEMON runs: one process driving all GPUs through b200probe_nvlink_a2a.  Rank 0 alone; the other ranks
        # wait on a CPU-side barrier so that nothing of theirs sits on the SMs the exchange kernels need.
        D.host_barrier()
        if rank == 0:
            nvlink["plugin_entry"] = nvlink_plugin_entry(p, world)
        D.host_barrier()

    # ---- rank 0 extras: read/write legs, host-buffer round trip, CPU baseline ---------------------
    line = None
    if rank == 0:
        def timed(fn, n=20):
            for _ in range(3):
                fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n
        rd = nbytes / timed(lambda: p.hbm_read(local_rank, src.data_ptr(), nbytes, part.data_ptr(), stream)) / 1e6
        wr = nbytes / timed(lambda: p.hbm_fill(local_rank, dst.data_ptr(), nbytes, seed, stream)) / 1e6
        import numpy as np

        hb = 256 << 20
        hsrc, hdst = p.host_alloc(hb), p.host_alloc(hb)          # pinned (b200probe_host_alloc)
        hsrc.view(np.uint32)[:] = np.arange(hb // 4, dtype=np.uint32)
        p.hbm_copy_host(local_rank, hsrc, hdst)
        t0 = time.perf_counter()
        for _ in range(5):
            hsum = p.hbm_copy_host(local_rank, hsrc, hdst)
        hostbuf_gbs = 5 * 2.0 * hb / (time.perf_counter() - t0) / 1e9
        hostbuf_ok = bool(np.array_equal(hsrc, hdst)) and hsum[0] == int(hsrc.view(np.uint32).sum(dtype=np.uint64))
        p.host_free(hsrc)
        p.host_free(hdst)
        p.lib.b200probe_hbm_release(local_rank)

        peaks, peak_src = measured_peaks()
        gemm = None
        if not args.no_gemm:
            try:                                   # a side leg must never cost the line: its failure is reported inside it
                gemm = gemm_leg(torch, p, local_rank, nvml_index, peaks, ClockSampler(nvml_index))
            except Exception as e:  # noqa: BLE001
                gemm = {"bound": "tensor", "error": str(e)[:300]}
        probe_round = None if args.no_probe_round else probe_round_leg(p)
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                traffic = json.load(f).get("hbm_ring_kernel_copy_1GiB_dram_bytes")
        except (OSError, ValueError):
            pass
        cpu = None
        parity = None
        if world == 1 and not args.no_cpu_baseline:
            _, o = load_oracle()
            cores = o.oracle_allowed_cpus()
            gbs, reps, dt, chk = cpu_copy_sample(o, cores, GIB, 12.0)
            cpu = {"value": round(gbs, 2), "unit": "GB/s", "cores": cores, "kind": "port", "cpu_model": cpu_model(),
                   "sample": f"oracle port of the copy pass over 1 GiB of host memory, {reps} passes in {dt:.1f} s, {cores} pthreads each pinned to one CPU",
                   "reference_path_nvml": nvml_poll_timing(o)}
            parity = chk == got
        achieved = 2.0 * nbytes / (launch_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": round(agg["gbs"], 2), "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(agg["ms"] / args.steps, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "bytes_per_step_per_gpu": 2 * nbytes, "buffer": "1 GiB src + 1 GiB dst resident in HBM",
                       "l2": "inputs 16x larger than the 126.5 MiB L2; no flush needed", "parallelism": f"replicas x{world} (no data-path collective)",
                       "kernel": "hbm_ring_kernel<COPY> (cp.async.bulk ring, 8 KiB x 4 stages x 2 warps, 1 CTA/SM)"},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": round(achieved / peaks["hbm_gbs"], 4), "traffic": traffic, "peak_source": peak_src,
                         "frac_of_nominal_8000": round(achieved / 8000.0, 4), "frac_of_bus_7672": round(achieved / 7672.0, 4),
                         "kernel": "hbm_ring_kernel<COPY>", "algorithmic_bytes_per_launch": 2 * nbytes,
                         "launch_ms": round(launch_ms, 5), "rank": 0},
            "e2e": {"value": round(e2e["gbs"], 2), "unit": "GB/s", "h2d_bytes_per_step": C.sizeof(L.HbmCfg) + 32, "d2h_bytes_per_step": 32,
                    "steps": e2e_steps, "ms_per_step": round(e2e["ms"] / e2e_steps, 4), "verified_every_step": bool(ok),
                    "what": "b200probe_hbm_sweep(cfg on host) -> memset dst, copy kernel, device-side verify + checksum, D2H verdict; wall clock",
                    "hostbuf_value": round(hostbuf_gbs, 2),
                    "hostbuf_what": "the same copy pass carrying HOST data (rank 0): pinned src -> H2D -> copy kernel + checksum -> D2H, 256 MiB each way per step; PCIe-bound (see e2e_hostbuf)"},
            "e2e_hostbuf": {"value": round(hostbuf_gbs, 2), "unit": "GB/s", "h2d_bytes_per_step": hb, "d2h_bytes_per_step": hb,
                            "roundtrip_identical": hostbuf_ok,
                            "what": "b200probe_hbm_copy_host: pinned host src -> H2D -> copy kernel + checksum -> D2H host dst, 8 MiB chunks pipelined on 3 streams (PCIe-bound: 2N bytes counted, N each way)"},
            "gpu_launches": args.steps * world,
            "clocks": clocks,
            "hbm_read_gbs": round(rd, 1), "hbm_write_gbs": round(wr, 1),
            "hbm_sustained": {"value": round(sustained["gbs"], 2), "unit": "GB/s", "seconds": round(sustained["ms"] / 1e3, 3), "launches_per_rank": sus_n,
                              "what": "the same copy launch back to back for >= 1 s after the timed K steps (aggregate over ranks, max-over-ranks time)"},
            "parity": {"dst_checksum_matches_oracle": parity, "sum64": f"{got[0]:#x}", "xor32": f"{got[1]:#x}"},
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if gemm:
            line["roofline_gemm"] = gemm
        if probe_round:
            line["probe_round"] = probe_round
        if nvlink:
            line["nvlink"] = nvlink
            ce = (nvlink.get("plugin_entry") or {}).get("copy_engines") or {}
            line["roofline_nvlink"] = {
                "bound": "nvlink", "achieved": nvlink["gbs_per_gpu_per_direction"], "peak": NVLINK_NOMINAL, "unit": "GB/s per direction per GPU",
                "frac": round(nvlink["gbs_per_gpu_per_direction"] / NVLINK_NOMINAL, 4), "peak_source": "nominal 18 links x 50 GB/s (no NVLink figure in MEASURED_PEAKS.json)",
                "measured_two_way_copy_engine_gbs": ce.get("gbs_per_gpu_per_direction"),
                "frac_of_measured_two_way_copy": (round(nvlink["gbs_per_gpu_per_direction"] / ce["gbs_per_gpu_per_direction"], 4) if ce.get("gbs_per_gpu_per_direction") else None),
                "guide_one_way_peer_copy_gbs": NVLINK_GUIDE_ONE_WAY, "kernel": nvlink["kernel"],
                "algorithmic_bytes_per_launch": nvlink["algorithmic_bytes_per_gpu_per_direction"], "traffic": None}
    if outputs:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
    if rank == 0:
        emit(line)
    # CPU-side wait: an NCCL barrier would park a spinning kernel on every waiting rank's GPU for as long as rank 0 works on its
    # extras, and rank 0's probe round drives ALL GPUs from one process — its kernels would be time-sliced against those kernels
    # (first seen as gpu0 "egress 234 GB/s": GPU 0 waiting 2 ms at the first step barrier for peers that had no time slice yet)
    D.host_barrier()
    p.close()
    if world > 1:
        import torch.distributed as td

        td.destroy_process_group()
    return 0


DUMP_WORDS = 1 << 22       # 4 Mi words of dst, 32 MiB as float64


def last_step_outputs(torch, p, ordinal, dst, stream):
    """What the timed copy handed its caller in the last step: dst (1 GiB), as the 32-bit words at a fixed seeded
    sample of positions, and the sum64 / xor32 checksum of the whole buffer from the device, split into exact
    32-bit halves.  float64 holds every uint32 exactly."""
    import numpy as np

    idx = np.sort(np.random.default_rng(0xB200).integers(0, dst.numel() // 4, DUMP_WORDS))
    words = dst.view(torch.int32)[torch.from_numpy(idx).to(dst.device)].to(torch.int64) & 0xFFFFFFFF
    part = torch.zeros(4, dtype=torch.int64, device=dst.device)
    p.hbm_read(ordinal, dst.data_ptr(), dst.numel(), part.data_ptr(), stream)
    torch.cuda.synchronize()
    s, x = part[0].item() & 0xFFFFFFFFFFFFFFFF, part[1].item() & 0xFFFFFFFF
    return {"dst_words_sample": words.cpu().numpy().astype(np.float64),
            "dst_checksum": np.array([s & 0xFFFFFFFF, s >> 32, x], dtype=np.float64)}


def nvlink_exchange(torch, D, p, local_rank, rank, world, stream, args):
    """configs[2]: every rank owns a window [recv world x S][send world x S]; handles are exchanged
    over torch.distributed (control data only) and every rank PUSHES its chunks into its peers' recv
    slots over NVLink with our TMA kernel (pushes beat pulls when both directions are loaded), one peer
    per step with a device-side step barrier; device-timed, max over ranks; landed data verified."""
    S = 256 << 20
    lib = p.lib
    seed = 0xB200
    win = C.c_void_p()
    handle = C.create_string_buffer(64)
    p._check(lib.b200probe_a2a_window_create(local_rank, world, S, C.byref(win), handle), "a2a_window_create")
    p._check(lib.b200probe_a2a_window_fill(local_rank, win, rank, world, S, seed, stream), "a2a_window_fill")
    torch.cuda.synchronize()
    handles = D.all_gather_bytes(handle.raw)
    peers = (C.c_void_p * world)()
    for r in range(world):
        if r == rank:
            peers[r] = win.value
        else:
            q = C.c_void_p()
            p._check(lib.b200probe_a2a_window_import(local_rank, handles[r], C.byref(q)), "a2a_window_import")
            peers[r] = q.value
    D.barrier()                      # every send half is filled before anyone pulls
    steps = max(3, min(args.steps, 20))

    def exchange(only_peer=-2):
        p._check(lib.b200probe_a2a_exchange(local_rank, rank, world, peers, S, seed, A2A_VARIANT, 0, only_peer, stream), "a2a_exchange")

    for _ in range(3):
        exchange()
    torch.cuda.synchronize()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        exchange()
    e1.record()
    torch.cuda.synchronize()
    D.barrier()
    ms = D.reduce_scalar(e0.elapsed_time(e1), "max") / steps
    exchange(-1)                     # complete the window (local slot) for verification
    torch.cuda.synchronize()
    D.barrier()
    # verify what landed here: recv slot r must hold pattern(chunk_seed(seed, r, rank))
    ok = 1.0
    part = torch.zeros(4, dtype=torch.int64, device=torch.device("cuda", local_rank))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle

    o = _oracle.load()
    for r in range(world):
        part.zero_()
        p.hbm_read(local_rank, win.value + r * S, S, part.data_ptr(), stream)
        torch.cuda.synchronize()
        got = (part[0].item() & 0xFFFFFFFFFFFFFFFF, part[1].item() & 0xFFFFFFFF)
        want = _oracle.pattern_checksum(o, S // 4, o.oracle_a2a_chunk_seed(seed, r, rank))
        if got != want:
            ok = 0.0
    ok = D.reduce_scalar(ok, "min")
    D.barrier()
    for r in range(world):
        if r != rank:
            lib.b200probe_a2a_window_release(local_rank, peers[r], 1)
    D.barrier()
    lib.b200probe_a2a_window_release(local_rank, win, 0)
    per_dir = (world - 1) * S / (ms * 1e-3) / 1e9
    push = "a2a_ring_kernel PUSH_TMA (pattern in smem, cp.async.bulk stores into IPC peer-mapped windows)"
    sync = ("a2a_stagger_kernel PUSH_SYNC (pattern in smem, cp.async.bulk stores into IPC peer-mapped windows; peers visited one at a "
            "time, rank r -> (r+t) mod G, with a device-side barrier over NVLink flags before every step)")
    names = {0: sync if world > 2 else push, 7: sync, 6: "a2a_stagger_kernel PUSH_STAGGER (no step barrier)", 5: "a2a_ring_kernel MIX_TMA", 1: "a2a_ring_kernel PULL_TMA (cp.async.bulk loads from IPC peer-mapped windows, bulk stores to local HBM)", 2: push,
             3: "a2a_direct_kernel PUSH_DIRECT (16-byte stores on peer pointers)", 4: "a2a_ring_kernel PUSH_BUF"}
    return {"bytes_per_pair": S, "ms_per_exchange": round(ms, 4), "gbs_per_gpu_per_direction": round(per_dir, 1),
            "aggregate_gbs": round(per_dir * world, 1), "frac_of_nominal_900": round(per_dir / NVLINK_NOMINAL, 4),
            "verified": bool(ok), "steps": steps,
            "kernel": names.get(A2A_VARIANT, str(A2A_VARIANT)), "algorithmic_bytes_per_gpu_per_direction": (world - 1) * S,
            "scaling": "every rank moves (world-1)*S per exchange: total work grows with N"}


def nvlink_plugin_entry(p, world):
    """Rank 0, single process, all GPUs: b200probe_nvlink_a2a exactly as the plugin's active-probe round calls it (PEER_ALL,
    verify), then the copy-engine leg (cudaMemcpyPeerAsync both ways) as the measured two-way peer-copy denominator."""
    from k3s_nvidia_b200 import _lib as L

    S = 256 << 20
    ords = list(range(world))
    out = {"bytes_per_pair": S, "gpus": world}
    try:
        t0 = time.perf_counter()
        rep = p.nvlink_a2a(ords, bytes_per_pair=S, warmup=2, reps=5, verify=1)
        wall = time.perf_counter() - t0
        src = {L.PAIR_SHARE: "share of the concurrent exchange", L.PAIR_ISOLATED: "isolated pairs", L.PAIR_STEPPED: "drained, device-stamped steps (one pair per rank per step)"}
        out.update({"gbs_per_gpu_per_direction": round(min(rep.egress_gbs[:world]), 1), "egress_min_max": [round(min(rep.egress_gbs[:world]), 1), round(max(rep.egress_gbs[:world]), 1)],
                    "ms_median": round(rep.ms_median, 4), "pair_min": round(rep.min_pair_gbs, 1), "pair_max": round(rep.max_pair_gbs, 1),
                    "pair_source": src.get(rep.pair_source, str(rep.pair_source)), "pair_max_le_900": rep.max_pair_gbs <= 900.0,
                    "verified": rep.verified == 1, "call_wall_s": round(wall, 3)})
        ce = p.nvlink_a2a(ords, bytes_per_pair=S, mode=L.A2A_CE, warmup=1, reps=5, verify=1)
        out["copy_engines"] = {"gbs_per_gpu_per_direction": round(min(ce.egress_gbs[:world]), 1), "ms_median": round(ce.ms_median, 4), "verified": ce.verified == 1,
                               "what": "cudaMemcpyPeerAsync of every chunk, all GPUs sending and receiving at once, same windows, same run"}
    except Exception as e:  # noqa: BLE001
        out["error"] = str(e)[:300]
    finally:
        try:
            p.a2a_release()
        except Exception:  # noqa: BLE001
            pass
    return out


def gemm_leg(torch, p, ordinal, nvml_index, peaks, sampler):
    """tcgen05 GEMM probe at 8192^3 for BOTH operand classes, and cuBLAS (torch.matmul) on the SAME device buffers in the
    same process: burst = median / best of 10 single launches, sustained = back to back for 4 s (MEASURED_PEAKS.json's
    protocol).  Data check: the library's own sampled fp64 check per class, and our C against cuBLAS's C on identical data."""
    from k3s_nvidia_b200 import _lib as L

    M = N = K = 8192
    dev = torch.device("cuda", ordinal)
    st = torch.cuda.current_stream().cuda_stream
    A = torch.empty(M * K, dtype=torch.int16, device=dev)
    B = torch.empty(N * K, dtype=torch.int16, device=dev)
    Cm = torch.empty(M * N, dtype=torch.int16, device=dev)
    Cl = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
    Ab, Bb = A.view(torch.bfloat16).view(M, K), B.view(torch.bfloat16).view(N, K)
    flop = 2.0 * M * N * K

    def ours():
        p._check(p.lib.b200probe_gemm_launch(ordinal, A.data_ptr(), B.data_ptr(), Cm.data_ptr(), M, N, K, st), "gemm_launch")

    def cublas():
        torch.matmul(Ab, Bb.t(), out=Cl)

    def burst(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(10):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        return flop / (statistics.median(ts) * 1e-3) / 1e12, flop / (min(ts) * 1e-3) / 1e12

    def sustained(fn, seconds=4.0):
        tot_ms, n = 0.0, 0
        while tot_ms < seconds * 1e3:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(100):
                fn()
            b.record()
            b.synchronize()
            tot_ms += a.elapsed_time(b)
            n += 100
        return flop * n / (tot_ms * 1e-3) / 1e12

    out = {"bound": "tensor", "unit": "TFLOP/s", "shape": [M, N, K], "peak": peaks.get("bf16_tflops"), "peak_sustained": peaks.get("bf16_tflops_sustained"),
           "kernel": "gemm_bf16_tn_2cta_kernel (tcgen05.mma cta_group::2, TMA loads, TMEM accumulators, TMA-store epilogue)",
           "algorithmic_flop_per_launch": flop, "protocol": "burst: 10 single launches after 3 warm-ups (median, best); sustained: back to back for 4 s", "classes": {}}
    for cls, name in ((L.GEMM_EXACT, "exact_k_over_128"), (L.GEMM_UNIFORM, "uniform_philox")):
        p._check(p.lib.b200probe_gemm_fill(ordinal, A.data_ptr(), M * K, 0xB200, 0 | (cls << 1), st), "gemm_fill")
        p._check(p.lib.b200probe_gemm_fill(ordinal, B.data_ptr(), N * K, 0xB200, 1 | (cls << 1), st), "gemm_fill")
        torch.cuda.synchronize()
        med, best = burst(ours)
        lmed, lbest = burst(cublas)
        sampler.start()
        sus = sustained(ours)
        sampler.stop()
        clk = sampler.summary()
        sampler.reasons.clear()
        lsus = sustained(cublas)
        ours()
        cublas()
        torch.cuda.synchronize()
        diff = (Cm.view(torch.bfloat16).view(M, N).float() - Cl.float()).abs()
        chk = p.gemm(nvml_index, warmup=1, reps=3, operands=cls)          # the library's own check (1024 samples vs fp64) on this class
        out["classes"][name] = {
            "ours": {"median": round(med, 1), "best": round(best, 1), "sustained_4s": round(sus, 1)},
            "cublas_same_buffers": {"median": round(lmed, 1), "best": round(lbest, 1), "sustained_4s": round(lsus, 1)},
            "ours_over_cublas": {"median": round(med / lmed, 4), "sustained_4s": round(sus / lsus, 4)},
            "frac_of_measured_burst": round(med / peaks["bf16_tflops"], 4) if peaks.get("bf16_tflops") else None,
            "frac_of_measured_sustained": round(sus / peaks["bf16_tflops_sustained"], 4) if peaks.get("bf16_tflops_sustained") else None,
            "frac_of_nominal_2250": round(med / 2250.0, 4),
            "clocks_during_sustained": clk,
            "data": {"library_check_verified": chk.verified == 1, "samples": chk.samples, "bad": chk.bad, "max_err_over_tol": round(chk.max_err_over_tol, 4),
                     "max_abs_diff_vs_cublas": float(diff.max().item()), "bit_identical_to_cublas": bool((diff == 0).all().item())},
        }
    p.lib.b200probe_gemm_release(ordinal)
    u = out["classes"]["uniform_philox"]
    out["achieved"] = u["ours"]["median"]                     # headline: SURVEY.md §8d's operand class
    out["frac"] = u["frac_of_measured_burst"]
    out["achieved_sustained"] = u["ours"]["sustained_4s"]
    out["frac_sustained"] = u["frac_of_measured_sustained"]
    return out


def probe_round_leg(p):
    """Wall time of ONE full active-probe round as the plugin daemon runs it (labels.ActiveProbeRunner.run_once: HBM sweep
    256 MiB-1 GiB x 3 modes, GEMM 8192^3, passive NVLink status and, with >= 2 GPUs, the exchange; labels written to a
    temporary features.d), cold (arenas allocated inside) and warm (second round)."""
    import tempfile

    from k3s_nvidia_b200.labels import ActiveProbeRunner, PREFIX

    out = {}
    os.environ["B200PROBE_IGNORE_TENANTS"] = "1"      # this bench has just loaded the GPU: to the runner it would look like a tenant
    try:
        with tempfile.TemporaryDirectory() as d:
            r = ActiveProbeRunner(p, features_dir=d, keep_arenas=True)
            t0 = time.perf_counter()
            labels = r.run_once()
            out["cold_s"] = round(time.perf_counter() - t0, 3)
            t0 = time.perf_counter()
            labels = r.run_once()
            out["warm_s"] = round(time.perf_counter() - t0, 3)
            r.release()
            out["gpus"] = p.device_count()
            out["labels"] = len(labels)
            out["gate"] = labels.get(f"{PREFIX}healthy")
            out["nvlink_egress_labels"] = {k[len(PREFIX):]: v for k, v in sorted(labels.items()) if k.endswith("nvlink-egress-gbs")}
            out["not_true"] = sorted(k[len(PREFIX):] + "=" + v for k, v in labels.items() if v == "false" or k.endswith("probe-state") and v != "probed")
            out["what"] = "labels.ActiveProbeRunner.run_once(): busy query, HBM sweep 256 MiB-1 GiB x 3 modes, GEMM 8192^3, passive NVLink, exchange (>= 2 GPUs), labels written"
    except Exception as e:  # noqa: BLE001
        out["error"] = str(e)[:300]
    finally:
        os.environ.pop("B200PROBE_IGNORE_TENANTS", None)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gemm", action="store_true", help="skip the GEMM roofline leg (about 20 s)")
    ap.add_argument("--no-probe-round", action="store_true", help="skip timing one full active-probe round")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
