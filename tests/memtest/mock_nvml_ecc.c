/*
 * mock_nvml_ecc.c — the mock NVML of tests/mock_nvml plus the three queries of the HBM integrity probe (TEST INFRASTRUCTURE).
 *
 * Environment, read at every query so a test can change it between calls:
 *   MOCK_NVML_ECC=d:mode:corrected:uncorrected,..      nvmlDeviceGetEccMode (1 enabled, 0 disabled) and the volatile totals
 *                                                      of nvmlDeviceGetTotalEccErrors for device d; a value of -1 makes that
 *                                                      query return NOT_SUPPORTED
 *   MOCK_NVML_REMAP=d:corr_rows:unc_rows:pending:failure,..   nvmlDeviceGetRemappedRows for device d
 * A device that is not listed answers NOT_SUPPORTED, as a part without ECC or row remapping does.
 */
#include "../mock_nvml/mock_nvml.c"

/* fields of device `dev` in the list `env` ("d:v1:v2:..,d:..."); returns 1 when the device is listed */
static int scripted(const char* env, int dev, long long* v, int nv) {
    const char* s = getenv(env);
    while (s && *s) {
        char* e;
        long d = strtol(s, &e, 10);
        int k = 0;
        while (*e == ':' && k < nv) v[k++] = strtoll(e + 1, &e, 10);
        if (d == dev && k == nv) return 1;
        s = strchr(e, ',');
        if (s) ++s;
    }
    return 0;
}

nvmlReturn_t nvmlDeviceGetEccMode(nvmlDevice_t d, nvmlEnableState_t* cur, nvmlEnableState_t* pend) {
    long long v[3];
    if (!scripted("MOCK_NVML_ECC", ((mdev_t*)d)->idx, v, 3) || v[0] < 0) return NVML_ERROR_NOT_SUPPORTED;
    *cur = *pend = v[0] ? NVML_FEATURE_ENABLED : NVML_FEATURE_DISABLED;
    return NVML_SUCCESS;
}

nvmlReturn_t nvmlDeviceGetTotalEccErrors(nvmlDevice_t d, nvmlMemoryErrorType_t type, nvmlEccCounterType_t counter, unsigned long long* count) {
    long long v[3];
    if (counter != NVML_VOLATILE_ECC) return NVML_ERROR_NOT_SUPPORTED;
    if (!scripted("MOCK_NVML_ECC", ((mdev_t*)d)->idx, v, 3)) return NVML_ERROR_NOT_SUPPORTED;
    const long long n = type == NVML_MEMORY_ERROR_TYPE_CORRECTED ? v[1] : v[2];
    if (n < 0) return NVML_ERROR_NOT_SUPPORTED;
    *count = (unsigned long long)n;
    return NVML_SUCCESS;
}

nvmlReturn_t nvmlDeviceGetRemappedRows(nvmlDevice_t d, unsigned int* corr, unsigned int* unc, unsigned int* pending, unsigned int* failure) {
    long long v[4];
    if (!scripted("MOCK_NVML_REMAP", ((mdev_t*)d)->idx, v, 4)) return NVML_ERROR_NOT_SUPPORTED;
    *corr = (unsigned)v[0]; *unc = (unsigned)v[1]; *pending = (unsigned)v[2]; *failure = (unsigned)v[3];
    return NVML_SUCCESS;
}
