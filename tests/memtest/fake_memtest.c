/*
 * fake_memtest.c — the probe interposer of tests/fake_probe plus a scripted b200probe_hbm_memtest (TEST INFRASTRUCTURE).
 *
 * Script, R = round number from 0 (rounds start when the runner asks b200probe_device_busy(0), as in fake_probe.c):
 *   FAKE_R<R>_MEMTEST = "i:bad:corr:unc:pending:failure,..."   result for NVML index i (-1 = not readable)
 *                       "i:enomem" / "i:cuda"                 B200PROBE_ENOMEM / a CUDA error (700, illegal address)
 * An index that is not listed gets a clean run: 160 GiB tested, no mismatch, ECC deltas 0, no pending or failed remap.
 */
#include "../fake_probe/fake_probe.c"

int b200probe_hbm_memtest(int idx, const b200probe_memtest_cfg_t* cfg, b200probe_memtest_result_t* out) {
    (void)cfg;
    memset(out, 0, sizeof(*out));
    out->bytes_tested = 160ull << 30;
    out->chunks = 160;
    out->passes = 1;
    out->first_bad_word = ~0ull;
    out->first_bad_element = -1;
    out->ecc_after.ecc_mode = 1;
    long long v[5] = {0, 0, 0, 0, 0};
    const char* s = script("MEMTEST");
    while (s && *s) {
        char* e;
        long i = strtol(s, &e, 10);
        if (i == idx && *e == ':') {
            if (!strncmp(e + 1, "enomem", 6)) return B200PROBE_ENOMEM;
            if (!strncmp(e + 1, "cuda", 4)) return B200PROBE_CUDA_BASE + 700;
            for (int k = 0; k < 5 && *e == ':'; ++k) v[k] = strtoll(e + 1, &e, 10);
        }
        s = strchr(e, ',');
        if (s) ++s;
    }
    out->bad_words = (uint64_t)v[0];
    if (v[0]) { out->first_bad_word = 12345; out->first_bad_element = 1; out->bad_bits = 4; }
    out->ecc_corrected_delta = v[1];
    out->ecc_uncorrected_delta = v[2];
    out->ecc_after.remap_pending = (int)v[3];
    out->ecc_after.remap_failure = (int)v[4];
    return 0;
}
