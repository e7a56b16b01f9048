/*
 * fake_gemm_fp8.c — the probe interposer of tests/fake_probe plus a scripted b200probe_gemm_fp8 (TEST INFRASTRUCTURE).
 *
 * Script, R = round number from 0 (rounds start when the runner asks b200probe_device_busy(0), as in fake_probe.c):
 *   FAKE_R<R>_FP8 = "i:tflops,..."                    median TFLOP/s of NVML index i, data verified
 *                   "i:mismatch" / "i:enomem" / "i:cuda"   B200PROBE_EMISMATCH / B200PROBE_ENOMEM / a CUDA error (700)
 * An index that is not listed gets a clean run at 3000 TFLOP/s.
 */
#include "../fake_probe/fake_probe.c"

int b200probe_gemm_fp8(int idx, const b200probe_gemm_cfg_t* cfg, b200probe_gemm_result_t* out) {
    (void)cfg;
    memset(out, 0, sizeof(*out));
    out->m = out->n = out->k = 8192; out->samples = 1024; out->verified = 1;
    double tflops = 3000.0;
    const char* s = script("FP8");
    while (s && *s) {
        char* e;
        long i = strtol(s, &e, 10);
        if (i == idx && *e == ':') {
            if (!strncmp(e + 1, "mismatch", 8)) { out->verified = 0; out->bad = 3; return B200PROBE_EMISMATCH; }
            if (!strncmp(e + 1, "enomem", 6)) { out->verified = -1; return B200PROBE_ENOMEM; }
            if (!strncmp(e + 1, "cuda", 4)) { out->verified = -1; return B200PROBE_CUDA_BASE + 700; }
            tflops = strtod(e + 1, &e);
        }
        s = strchr(e, ',');
        if (s) ++s;
    }
    out->tflops_median = tflops; out->tflops_best = tflops * 1.01;
    out->ms_median = 2.0 * 8192.0 * 8192.0 * 8192.0 / (tflops * 1e9);
    return 0;
}
