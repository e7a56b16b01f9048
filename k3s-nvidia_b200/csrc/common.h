// Internal helpers shared by the translation units of libb200probe.so.  Not part of the ABI.
#pragma once
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include "../../include/b200probe.h"

namespace b200 {

// thread-local detailed error text (b200probe_last_error)
void set_error(const char* fmt, ...) __attribute__((format(printf, 1, 2)));
const char* get_error();

// NVML index -> CUDA ordinal (by UUID); initialises CUDA lazily.  Returns a b200probe rc.
int cuda_ordinal_of(int nvml_idx, int* ordinal);
// Make sure CUDA is usable and `ordinal` is an sm_100 device; caches per-device properties.
struct DevProps {
    int  sms;
    int  l2_bytes;
    int  smem_optin;
    int  cc_major, cc_minor;
};
int device_props(int ordinal, DevProps* out);

// Device-side check of a buffer against the closed-form pattern (hbm_sweep.cu): checksum + count of
// words that differ.  d_partials = 4 x u64 scratch on the device; synchronises `stream`.
struct VerifyResult { uint64_t sum; uint32_t x; uint64_t bad, first; };
int verify_pattern(int ordinal, const void* buf, uint64_t bytes, uint32_t seed, unsigned long long* d_partials, void* stream, VerifyResult* out);

inline int cuda_rc(int cuda_err) { return cuda_err == 0 ? 0 : B200PROBE_CUDA_BASE + cuda_err; }

}  // namespace b200

#define B200_CUDA_TRY(expr)                                                                   \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            b200::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
            return b200::cuda_rc((int)e__);                                                   \
        }                                                                                     \
    } while (0)

// A failed cudaMalloc is a RESOURCE verdict (a tenant holds the memory), not a CUDA fault: the host must be able to tell
// the two apart (B200PROBE_ENOMEM -> "inconclusive", never "unhealthy").
#define B200_ALLOC_TRY(expr)                                                                                  \
    do {                                                                                                      \
        cudaError_t e__ = (expr);                                                                             \
        if (e__ == cudaErrorMemoryAllocation) { cudaGetLastError(); b200::set_error("%s: out of device memory", #expr); return B200PROBE_ENOMEM; } \
        if (e__ != cudaSuccess) { b200::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); return b200::cuda_rc((int)e__); } \
    } while (0)

// ---- data pattern, shared host/device (header-only so the kernels inline it) -----------------
#if defined(__CUDACC__)
#define B200_HD __host__ __device__ __forceinline__
#else
#define B200_HD inline
#endif
B200_HD uint32_t b200_pattern_word(uint64_t i, uint32_t seed) {
    return ((uint32_t)i * 2654435761u) ^ seed ^ (uint32_t)(i >> 32);
}
// splitmix-style 32-bit finaliser (GEMM operand generator)
B200_HD uint32_t b200_mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
// ---- GEMM operand class 1 (SURVEY.md §8d "GEMM probe": bf16 A,B ~ U(-1,1) from Philox seed 0xB200) ----------------
// Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123
// reference constants).  Counter-based: word j of block b is a pure function of (b, key), so the device fill, the
// host-side check and the oracle agree without sharing state.
B200_HD void b200_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// element e of matrix `which` (0 = A, 1 = B): word e%4 of Philox block (e/4, which, 0) under key (seed, 0);
// u = top 24 bits -> x = u * 2^-23 - 1 in [-1, 1) (exact in fp32) -> bf16 round-to-nearest-even.  The E4M3 UNIFORM class
// rounds the same x to E4M3 instead.
B200_HD float b200_gemm_uniform_f32(uint64_t e, uint32_t seed, int which) {
    uint32_t r[4];
    const uint64_t blk = e >> 2;
    b200_philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)which, 0u, seed, 0u, r);
    return (float)(r[e & 3] >> 8) * (1.0f / 8388608.0f) - 1.0f;
}
B200_HD uint16_t b200_gemm_uniform_bits(uint64_t e, uint32_t seed, int which) {
    const float x = b200_gemm_uniform_f32(e, seed, which);
    uint32_t u;
#if defined(__CUDA_ARCH__)
    u = __float_as_uint(x);
#else
    memcpy(&u, &x, 4);
#endif
    return (uint16_t)((u + 0x7fffu + ((u >> 16) & 1u)) >> 16);
}

// bf16 operand element e of matrix `which`: k/128 with k an integer in [-128,127], exactly
// representable in bf16 (8 significant bits), so the CPU oracle and the device agree on the bits.
B200_HD uint32_t b200_gemm_elem_hash(uint64_t e, uint32_t seed, int which) {
    return b200_mix32((uint32_t)e * 0x9E3779B1u ^ b200_mix32(seed + 0x51ED27u * (uint32_t)(which + 1)) ^ (uint32_t)(e >> 32));
}
B200_HD uint16_t b200_gemm_elem_bits(uint64_t e, uint32_t seed, int which) {
    uint32_t h = b200_gemm_elem_hash(e, seed, which);
    int k = (int)(h & 0xFF) - 128;                    // [-128,127]
    float f = (float)k * (1.0f / 128.0f);             // exact
    uint32_t u;
#if defined(__CUDA_ARCH__)
    u = __float_as_uint(f);
#else
    memcpy(&u, &f, 4);
#endif
    return (uint16_t)(u >> 16);                       // exact: low 16 mantissa bits are zero
}

// ---- E4M3 operands (kind::f8f6f4): one byte per element, sign | 4-bit exponent (bias 7) | 3-bit mantissa, max 448 ----------
// fp32 -> E4M3 with round-to-nearest-even, saturating to +-448 (NaN -> 0x7F): the host twin of cvt.rn.satfinite.e4m3x2.f32.
B200_HD uint8_t b200_e4m3_rne(float x) {
    uint32_t u;
#if defined(__CUDA_ARCH__)
    u = __float_as_uint(x);
#else
    memcpy(&u, &x, 4);
#endif
    const uint8_t s = (uint8_t)((u >> 24) & 0x80u);
    u &= 0x7fffffffu;
    if (u > 0x7f800000u) return (uint8_t)(s | 0x7f);
    if (u >= 0x43E00000u) return (uint8_t)(s | 0x7e);            // |x| >= 448: saturate
    if (u < 0x3C800000u) {                                      // |x| < 2^-6: subnormal, multiples of 2^-9 (8 = the smallest normal)
        float a;
#if defined(__CUDA_ARCH__)
        a = __uint_as_float(u);
#else
        memcpy(&a, &u, 4);
#endif
        return (uint8_t)(s | (uint8_t)rintf(a * 512.0f));
    }
    u += 0x7ffffu + ((u >> 20) & 1u);                            // keep 3 mantissa bits, ties to even (a carry bumps the exponent)
    return (uint8_t)(s | (uint8_t)((u >> 20) - (120u << 3)));     // rebias the exponent from 127 to 7
}
// E4M3 operand element e of matrix `which` (0 = A, 1 = B).
//   EXACT    the integer (h & 0xF) - 8 in [-8, 7] with h the bf16 EXACT class's hash: every such integer is an E4M3 value,
//            products are at most 64 in magnitude, so every partial sum of up to 2^18 terms is an exact fp32 integer
//   UNIFORM  the bf16 UNIFORM class's fp32 Philox value in [-1, 1), rounded to E4M3 (never saturates)
B200_HD float b200_gemm_e4m3_value(uint64_t e, uint32_t seed, int which, int uniform) {
    return uniform ? b200_gemm_uniform_f32(e, seed, which) : (float)((int)(b200_gemm_elem_hash(e, seed, which) & 0xF) - 8);
}
