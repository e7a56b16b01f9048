"""HBM integrity probe figures on one GPU, in one process: the card and its power limit, the rate of one verify+write march
element against the library's copy sweep at 1 GiB (kernel time from torch.profiler, and the whole synchronous call on the host clock), the
allocation and test time of the full-memory memtest at the default
fraction, and the wall time of one active-probe round with the memtest off and on.  Prints one JSON line.

    python tools/memtest_bench.py [--gpu 0] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(gpu):
    q = subprocess.run(["nvidia-smi", "-i", str(gpu), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    name, power, clock = (x.strip() for x in q.split(","))
    return name, power, clock


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch

    from k3s_nvidia_b200 import _lib as L
    from k3s_nvidia_b200 import labels
    from k3s_nvidia_b200.probe import Probe

    name, power, clock = card(args.gpu)
    p = Probe()
    idx = args.gpu
    ordinal = p.device_info(idx).cuda_ordinal if p.device_info(idx).cuda_ordinal >= 0 else args.gpu
    copy = p.hbm_sweep(idx, min_bytes=1 << 30, max_bytes=1 << 30, modes=L.HBM_COPY, warmup=3, reps=20, verify=0)[0].gbs_median
    p.release([ordinal])

    # one verify+write element on 1 GiB: kernel time from torch.profiler, and the host clock around the synchronous call
    from torch.profiler import ProfilerActivity, profile

    nbytes = 1 << 30
    buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{ordinal}")
    p.memtest_element(ordinal, buf.data_ptr(), nbytes, 0, L.MEMTEST_WRITE, 0, 0xB200)
    seed, ts = 0xB200, []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            t0 = time.perf_counter()
            p.memtest_element(ordinal, buf.data_ptr(), nbytes, 0, L.MEMTEST_VERIFY | L.MEMTEST_WRITE, seed, ~seed & 0xFFFFFFFF)
            ts.append(time.perf_counter() - t0)
            seed = ~seed & 0xFFFFFFFF
    ev = [e for e in prof.key_averages() if "hbm_memtest_kernel" in e.key][0]
    kernel_ms = (getattr(ev, "device_time_total", None) or ev.cuda_time_total) / ev.count / 1e3
    elem_kernel = 2 * nbytes / (kernel_ms * 1e-3) / 1e9
    elem_call = 2 * nbytes / float(np.median(ts)) / 1e9
    del buf
    torch.cuda.empty_cache()

    t0 = time.perf_counter()
    r = p.hbm_memtest(idx)
    call_ms = (time.perf_counter() - t0) * 1e3
    memtest = dict(call_ms=round(call_ms, 1), bytes_tested=r.bytes_tested, gib=round(r.bytes_tested / 2**30, 1), chunks=r.chunks, free_before=r.free_before, total=r.total,
                   alloc_ms=round(r.alloc_ms, 1), test_ms=round(r.test_ms, 1), gbs=round(r.gbs), bad_words=r.bad_words,
                   ecc_corrected_delta=r.ecc_corrected_delta, ecc_uncorrected_delta=r.ecc_uncorrected_delta, remap_pending=r.remap_pending,
                   remap_failure=r.remap_failure)

    os.environ["B200PROBE_IGNORE_TENANTS"] = "1"        # this process is the only tenant
    rounds = {}
    with tempfile.TemporaryDirectory() as d:
        for label, frac in (("off", None), ("on", "0.9"), ("off_again", None)):
            if frac is None:
                os.environ.pop("B200PROBE_MEMTEST_FRACTION", None)
            else:
                os.environ["B200PROBE_MEMTEST_FRACTION"] = frac
            runner = labels.ActiveProbeRunner(p, features_dir=os.path.join(d, label), interval_s=3600)
            t0 = time.perf_counter()
            got = runner.run_once()
            rounds[label] = dict(wall_s=round(time.perf_counter() - t0, 2), gate=got.get(labels.PREFIX + "healthy"),
                                 memtest_healthy=got.get(labels.PREFIX + f"gpu{idx}.hbm-memtest-healthy"))
    out = dict(card=name, power_limit=power, max_sm_clock=clock, gpu=idx, copy_sweep_1gib_gbs=round(copy),
               element_1gib_kernel_gbs=round(elem_kernel), element_1gib_over_copy=round(elem_kernel / copy, 3), element_1gib_call_gbs=round(elem_call),
               memtest=memtest, probe_round=rounds)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    p.close()


if __name__ == "__main__":
    main()
