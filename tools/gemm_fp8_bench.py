"""FP8 tensor-core probe figures on one GPU, in one process: the card, its power limit and SM clocks; for each E4M3 operand class
the library entry (burst median and best of 10, sustained for 4 s, data verdict), then our kernel and cuBLASLt FP8
(torch._scaled_mm, scales 1.0, bf16 out) on the SAME device buffers with the same protocol, their ratio and whether the two C
matrices are bit-identical; the bf16 probe for contrast; and the wall time of one active-probe round with the FP8 probe off
and on.  8192^3 unless --mnk says otherwise.  Prints one JSON line.

    python tools/gemm_fp8_bench.py [--gpu 0] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def smi(gpu, fields):
    q = subprocess.run(["nvidia-smi", "-i", str(gpu), f"--query-gpu={fields}", "--format=csv,noheader,nounits"], capture_output=True, text=True).stdout
    return [x.strip() for x in q.strip().split(",")]


class ClockSampler:
    """SM clock and board power every 0.25 s while a sustained run is in flight (read-only NVML queries through nvidia-smi)."""

    def __init__(self, gpu):
        self.gpu, self.samples, self._stop = gpu, [], threading.Event()

    def __enter__(self):
        def loop():
            while not self._stop.is_set():
                try:
                    clk, pw = smi(self.gpu, "clocks.sm,power.draw")
                    self.samples.append((float(clk), float(pw)))
                except (ValueError, IndexError):
                    pass
                self._stop.wait(0.25)
        self._t = threading.Thread(target=loop, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join()

    def summary(self):
        if not self.samples:
            return {}
        clk = sorted(s[0] for s in self.samples)
        pw = sorted(s[1] for s in self.samples)
        return dict(sm_mhz_median=clk[len(clk) // 2], sm_mhz_min=clk[0], power_w_median=pw[len(pw) // 2], samples=len(clk))


def timed(fn, flop, warmup=3, reps=10, sustain_s=4.0, gpu=0):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    med = 0.5 * (ms[len(ms) // 2 - 1] + ms[len(ms) // 2])
    batch = max(1, int(0.25 / (med * 1e-3)))
    total_ms, n = 0.0, 0
    with ClockSampler(gpu) as clk:
        while total_ms * 1e-3 < sustain_s:
            e0.record()
            for _ in range(batch):
                fn()
            e1.record()
            e1.synchronize()
            total_ms += e0.elapsed_time(e1)
            n += batch
    return dict(tflops_median=round(flop / (med * 1e-3) / 1e12, 1), tflops_best=round(flop / (ms[0] * 1e-3) / 1e12, 1),
                tflops_sustained=round(flop * n / (total_ms * 1e-3) / 1e12, 1), sustained_clocks=clk.summary())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--mnk", type=int, default=8192)
    ap.add_argument("--out")
    args = ap.parse_args()

    import torch

    from k3s_nvidia_b200 import _lib as L
    from k3s_nvidia_b200 import labels
    from k3s_nvidia_b200.probe import Probe

    name, power, max_clk, clk_now = smi(args.gpu, "name,power.limit,clocks.max.sm,clocks.sm")
    p = Probe()
    idx = args.gpu
    ordinal = p.device_info(idx).cuda_ordinal if p.device_info(idx).cuda_ordinal >= 0 else args.gpu
    torch.cuda.set_device(ordinal)
    m = n = k = args.mnk
    flop = 2.0 * m * n * k
    out = dict(card=name, power_limit_w=power, max_sm_clock_mhz=max_clk, sm_clock_idle_mhz=clk_now, gpu=idx, m=m, n=n, k=k)

    for cls, cname in ((L.GEMM_EXACT, "exact"), (L.GEMM_UNIFORM, "uniform")):
        with ClockSampler(args.gpu) as clk:
            r = p.gemm_fp8(idx, m=m, n=n, k=k, warmup=3, reps=10, sustain_seconds=4.0, operands=cls)
        entry = dict(tflops_median=round(r.tflops_median, 1), tflops_best=round(r.tflops_best, 1), tflops_sustained=round(r.tflops_sustained, 1),
                     verified=r.verified, bad=r.bad, samples=r.samples, max_err_over_tol=round(r.max_err_over_tol, 4), clocks=clk.summary())
        p.release([ordinal])

        dev = f"cuda:{ordinal}"
        st = torch.cuda.current_stream().cuda_stream
        a = torch.empty(m * k, dtype=torch.uint8, device=dev)
        b = torch.empty(n * k, dtype=torch.uint8, device=dev)
        p._check(p.lib.b200probe_gemm_fill(ordinal, a.data_ptr(), m * k, 0xB200, L.GEMM_FILL_E4M3 | (cls << 1) | 0, st), "gemm_fill A")
        p._check(p.lib.b200probe_gemm_fill(ordinal, b.data_ptr(), n * k, 0xB200, L.GEMM_FILL_E4M3 | (cls << 1) | 1, st), "gemm_fill B")
        c_ours = torch.empty(m, n, dtype=torch.bfloat16, device=dev)
        a8, b8 = a.view(torch.float8_e4m3fn).view(m, k), b.view(torch.float8_e4m3fn).view(n, k)
        one = torch.ones((), dtype=torch.float32, device=dev)
        ours = timed(lambda: p.gemm_fp8_launch(ordinal, a.data_ptr(), b.data_ptr(), c_ours.data_ptr(), m, n, k, st), flop, gpu=args.gpu)
        cublas = timed(lambda: torch._scaled_mm(a8, b8.t(), scale_a=one, scale_b=one, out_dtype=torch.bfloat16), flop, gpu=args.gpu)
        p.gemm_fp8_launch(ordinal, a.data_ptr(), b.data_ptr(), c_ours.data_ptr(), m, n, k, st)
        c_ref = torch._scaled_mm(a8, b8.t(), scale_a=one, scale_b=one, out_dtype=torch.bfloat16)
        torch.cuda.synchronize()
        differ = int((c_ours.view(torch.int16) != c_ref.view(torch.int16)).sum().item())
        out[cname] = dict(probe_entry=entry, our_kernel=ours, cublaslt_fp8=cublas,
                          ratio_median=round(ours["tflops_median"] / cublas["tflops_median"], 3),
                          ratio_sustained=round(ours["tflops_sustained"] / cublas["tflops_sustained"], 3),
                          c_bit_identical_to_cublas=differ == 0, c_elements_differing=differ)
        del a, b, c_ours, c_ref, a8, b8
        torch.cuda.empty_cache()

    bf = {}
    for cls, cname in ((L.GEMM_EXACT, "exact"), (L.GEMM_UNIFORM, "uniform")):
        r = p.gemm(idx, m=m, n=n, k=k, warmup=3, reps=10, operands=cls)
        bf[cname] = dict(tflops_median=round(r.tflops_median, 1), tflops_best=round(r.tflops_best, 1), verified=r.verified)
    p.release([ordinal])
    out["bf16_probe"] = bf

    os.environ["B200PROBE_IGNORE_TENANTS"] = "1"        # this process is the only tenant
    rounds = {}
    with tempfile.TemporaryDirectory() as d:
        for label, on in (("off", False), ("on", True), ("off_again", False)):
            if on:
                os.environ["B200PROBE_GEMM_FP8"] = "1"
            else:
                os.environ.pop("B200PROBE_GEMM_FP8", None)
            runner = labels.ActiveProbeRunner(p, features_dir=os.path.join(d, label), interval_s=3600)
            t0 = time.perf_counter()
            got = runner.run_once()
            rounds[label] = dict(wall_s=round(time.perf_counter() - t0, 2), gate=got.get(labels.PREFIX + "healthy"),
                                 fp8_tflops=got.get(labels.PREFIX + f"gpu{idx}.gemm-fp8-tflops"), fp8_healthy=got.get(labels.PREFIX + f"gpu{idx}.gemm-fp8-healthy"))
    out["probe_round"] = rounds
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(f"# tools/gemm_fp8_bench.py on one {name} (power limit {power} W, max SM clock {max_clk} MHz), one process, {m}x{n}x{k}.\n")
            f.write("# probe_entry = b200probe_gemm_fp8 (3 warm-up, 10 timed, 4 s sustained); our_kernel / cublaslt_fp8 = b200probe_gemm_fp8_launch and\n"
                    "# torch._scaled_mm (scales 1.0, bf16 out) on the same device buffers, CUDA events, same protocol; clocks sampled during the sustained run.\n")
            f.write(line + "\n")
    p.close()


if __name__ == "__main__":
    main()
