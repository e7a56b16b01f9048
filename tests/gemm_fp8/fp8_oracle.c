/*
 * fp8_oracle.c — CPU oracle of the E4M3 operand classes of the FP8 tensor-core probe (TEST INFRASTRUCTURE).
 * Restates include/b200probe.h's description independently of the library; only Philox4x32-10 comes from liboracle.
 *
 * E4M3 (OCP FP8 "e4m3fn"): sign | 4-bit exponent, bias 7 | 3-bit mantissa; no infinities, S.1111.111 is NaN, max 448.
 * Rounding is restated as a search: the representable value nearest to x, ties to the even code (mantissa bit 0 clear),
 * values beyond 448 saturate.
 *   EXACT    element e of matrix `which`: h = mix32(lo(e) * 0x9E3779B1 ^ mix32(seed + 0x51ED27 * (which + 1)) ^ hi(e)),
 *            value (h & 0xF) - 8, an integer in [-8, 7]
 *   UNIFORM  word e mod 4 of Philox block (e div 4, which, 0) under key (seed, 0), top 24 bits u: x = u / 2^23 - 1 in
 *            [-1, 1), rounded to E4M3
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

static uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

double oracle_e4m3_value(uint8_t v) {
    const int e = (v >> 3) & 15, m = v & 7;
    if (e == 15 && m == 7) return NAN;
    const double mag = e == 0 ? m / 8.0 * ldexp(1.0, -6) : (1.0 + m / 8.0) * ldexp(1.0, e - 7);
    return (v & 0x80) ? -mag : mag;
}

uint8_t oracle_e4m3_round(double x) {
    static double mag[0x7f];
    static int ready;
    if (!ready) { for (int c = 0; c < 0x7f; ++c) mag[c] = oracle_e4m3_value((uint8_t)c); ready = 1; }
    if (isnan(x)) return 0x7f;
    const uint8_t s = signbit(x) ? 0x80 : 0;
    const double a = fabs(x);
    int best = 0;
    for (int c = 1; c <= 0x7e; ++c) {
        const double dc = fabs(mag[c] - a), db = fabs(mag[best] - a);
        if (dc < db || (dc == db && (c & 1) == 0)) best = c;
    }
    return (uint8_t)(s | best);
}

float oracle_fp8_uniform_f32(uint64_t e, uint32_t seed, int which) {
    const uint64_t blk = e / 4;
    const uint32_t ctr[4] = {(uint32_t)(blk & 0xffffffffu), (uint32_t)(blk >> 32), (uint32_t)which, 0u}, key[2] = {seed, 0u};
    uint32_t r[4];
    oracle_philox4x32_10(ctr, key, r);
    return (float)((double)(r[e % 4] >> 8) / 8388608.0 - 1.0);
}

/* which: bit 0 = matrix (0 A, 1 B), bit 1 = class (0 EXACT, 1 UNIFORM) */
uint8_t oracle_fp8_operand(uint64_t e, uint32_t seed, int which) {
    const int mat = which & 1;
    if (which & 2) return oracle_e4m3_round(oracle_fp8_uniform_f32(e, seed, mat));
    const uint32_t h = mix32(((uint32_t)e * 0x9E3779B1u) ^ mix32(seed + 0x51ED27u * (uint32_t)(mat + 1)) ^ (uint32_t)(e >> 32));
    return oracle_e4m3_round((double)((int)(h & 0xF) - 8));
}

/* elements e0 .. e0 + n of one operand: E4M3 bytes, and (UNIFORM) the fp32 values before rounding */
void oracle_fp8_fill(uint8_t* dst, uint64_t e0, uint64_t n, uint32_t seed, int which) {
    for (uint64_t i = 0; i < n; ++i) dst[i] = oracle_fp8_operand(e0 + i, seed, which);
}
void oracle_fp8_uniform_f32_fill(float* dst, uint64_t e0, uint64_t n, uint32_t seed, int which) {
    for (uint64_t i = 0; i < n; ++i) dst[i] = oracle_fp8_uniform_f32(e0 + i, seed, which);
}

/* C[row][col] = sum_k A[row][k] * B[col][k] in fp64 (cls: 0 EXACT, 1 UNIFORM) */
double oracle_fp8_dot(int kdim, uint32_t seed, int cls, int row, int col) {
    double acc = 0.0;
    for (int k = 0; k < kdim; ++k)
        acc += oracle_e4m3_value(oracle_fp8_operand((uint64_t)row * kdim + k, seed, (cls << 1) | 0)) *
               oracle_e4m3_value(oracle_fp8_operand((uint64_t)col * kdim + k, seed, (cls << 1) | 1));
    return acc;
}
