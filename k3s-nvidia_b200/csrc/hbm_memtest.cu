// HBM integrity probe for sm_100a: a march test over the GPU's free memory (DESIGN.md §4.4).
//
// One kernel runs one march element over one buffer.  For every u32 word i it may compare the word with the
// closed-form pattern b200_pattern_word(base_word + i, expect_seed) and may then overwrite it in place with the
// pattern under write_seed.  base_word is the buffer's first word in the whole tested space, so the pattern is
// address-in-address across every chunk: two chunks that alias each other in HBM read back each other's words.
//
// Data path (the bulk-TMA ring of hbm_sweep.cu): every warp owns a ring of shared-memory stages; lane 0 brings a
// stage in with cp.async.bulk global->shared on an mbarrier, the lanes compare and overwrite the 16-byte words in
// the stage, fence.proxy.async hands the stage to the async proxy and lane 0 bulk-stores it back to the same
// address.  An element that only writes (E0) generates into the stages without loading them.
//
// Mismatches are counted on the device: number of words, lowest global word index, OR of got ^ want.
// Roofline: HBM bound.  Algorithmic bytes: verify N, write N, verify+write 2N.
#include <cuda_runtime.h>
#include <time.h>

#include <algorithm>
#include <vector>

#include "common.h"
#include "ptx.cuh"

namespace {

using namespace b200ptx;

// 4 warps x 4 stages x 8 KiB = 128 KiB of shared memory per CTA, one CTA per SM: a verify+write element runs at
// 0.93-0.94 x the copy sweep (profiles/memtest_bench_r01.txt)
constexpr int kWarps = 4;
constexpr int kStages = 4;
constexpr uint32_t kStageBytes = 8192;
constexpr uint32_t kSeed1Xor = 0x5A5A5A5Au;

struct MemtestArgs {
    uint8_t* buf;
    uint64_t bytes;                 // multiple of 4
    uint64_t base_word;
    int flags;                      // B200PROBE_MEMTEST_VERIFY | B200PROBE_MEMTEST_WRITE
    uint32_t expect_seed, write_seed;
    unsigned long long* res;        // [0] mismatching words, [1] lowest mismatching word, [2] OR of got ^ want
};

// b200_pattern_word(w0 + j, seed) ^ seed for the j-th word of a stage whose first global word is w0 = (hi:lo0).
// The high half of the index is carried per word, so a stage may straddle a 2^32-word boundary.
__device__ __forceinline__ uint32_t pattern_base(uint32_t lo0, uint32_t hi, uint32_t j) {
    const uint32_t lo = lo0 + j;
    return lo * 2654435761u ^ (hi + (lo < lo0 ? 1u : 0u));
}

struct Mismatch {
    unsigned long long bad = 0, first = ~0ull;
    uint32_t bits = 0;
    // one word: got vs want at global word index w
    __device__ __forceinline__ void word(uint32_t got, uint32_t want, unsigned long long w) {
        if (got != want) {
            ++bad;
            first = min(first, w);
            bits |= got ^ want;
        }
    }
    __device__ __forceinline__ void publish(unsigned long long* res) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            bad += __shfl_xor_sync(0xffffffffu, bad, o);
            first = min(first, (unsigned long long)__shfl_xor_sync(0xffffffffu, first, o));
            bits |= __shfl_xor_sync(0xffffffffu, bits, o);
        }
        if ((threadIdx.x & 31) == 0 && bad) {
            atomicAdd(res, bad);
            atomicMin(res + 1, first);
            atomicOr(res + 2, (unsigned long long)bits);
        }
    }
};

__global__ void __launch_bounds__(kWarps * 32) hbm_memtest_kernel(MemtestArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t full_bar[kWarps * kStages];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kWarps * kStages; ++i) mbar_init(smem_u32(&full_bar[i]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const bool verify = a.flags & B200PROBE_MEMTEST_VERIFY, write = a.flags & B200PROBE_MEMTEST_WRITE;
    const uint64_t bulk_bytes = a.bytes & ~15ull;
    const uint64_t nchunks = (bulk_bytes + kStageBytes - 1) / kStageBytes;
    const uint64_t worker = (uint64_t)blockIdx.x * kWarps + warp;
    const uint64_t nworkers = (uint64_t)gridDim.x * kWarps;
    const uint64_t n_my = worker < nchunks ? (nchunks - worker + nworkers - 1) / nworkers : 0;

    const uint32_t ring = smem_u32(smem) + warp * kStages * kStageBytes;
    uint8_t* ring_ptr = smem + (size_t)warp * kStages * kStageBytes;
    const uint32_t bar0 = smem_u32(&full_bar[warp * kStages]);
    const uint64_t pol = policy_evict_first();
    const uint32_t ws_x = a.write_seed, es_x = a.expect_seed;

    auto chunk_off = [&](uint64_t k) { return (worker + k * nworkers) * (uint64_t)kStageBytes; };
    auto chunk_len = [&](uint64_t k) { return (uint32_t)min((uint64_t)kStageBytes, bulk_bytes - chunk_off(k)); };
    uint32_t ps = 0, cs = 0, cph = 0;
    uint64_t issued = 0;
    auto load_next = [&]() {
        const uint32_t len = chunk_len(issued);
        mbar_expect_tx(bar0 + ps * 8, len);
        bulk_g2s(ring + ps * kStageBytes, a.buf + chunk_off(issued), len, bar0 + ps * 8, pol);
        ++issued;
        if (++ps == kStages) ps = 0;
    };
    auto advance = [&]() { if (++cs == kStages) { cs = 0; cph ^= 1; } };

    Mismatch mm;
    if (!verify) {
        // write only (E0): generate into the stage, bulk-store it; a stage is reused once its store has read it
        for (uint64_t k = 0; k < n_my; ++k) {
            if (k >= kStages) {
                if (lane == 0) bulk_wait_read<kStages - 1>();
                __syncwarp();
            }
            uint4* st = reinterpret_cast<uint4*>(ring_ptr + (size_t)cs * kStageBytes);
            const uint32_t nvec = chunk_len(k) >> 4;
            const uint64_t w0 = a.base_word + (chunk_off(k) >> 2);
            const uint32_t lo0 = (uint32_t)w0, hi = (uint32_t)(w0 >> 32);
#pragma unroll 4
            for (uint32_t i = lane; i < nvec; i += 32) {
                const uint32_t j = i * 4;
                st[i] = make_uint4(pattern_base(lo0, hi, j) ^ ws_x, pattern_base(lo0, hi, j + 1) ^ ws_x, pattern_base(lo0, hi, j + 2) ^ ws_x,
                                   pattern_base(lo0, hi, j + 3) ^ ws_x);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                bulk_s2g(a.buf + chunk_off(k), ring + cs * kStageBytes, chunk_len(k), pol);
                bulk_commit();
            }
            advance();
        }
    } else if (n_my > 0) {
        // verify (+ write back): up to kStages - 1 loads ahead when the stages are also stored, kStages when not
        const uint64_t depth = write ? kStages - 1 : kStages;
        if (lane == 0) {
            const uint64_t ahead = min(depth, n_my);
            while (issued < ahead) load_next();
        }
        for (uint64_t k = 0; k < n_my; ++k) {
            mbar_wait(bar0 + cs * 8, cph);
            uint4* st = reinterpret_cast<uint4*>(ring_ptr + (size_t)cs * kStageBytes);
            const uint32_t nvec = chunk_len(k) >> 4;
            const uint64_t w0 = a.base_word + (chunk_off(k) >> 2);
            const uint32_t lo0 = (uint32_t)w0, hi = (uint32_t)(w0 >> 32);
#pragma unroll 2
            for (uint32_t i = lane; i < nvec; i += 32) {
                const uint32_t j = i * 4;
                const uint4 v = st[i];
                const uint32_t f0 = pattern_base(lo0, hi, j), f1 = pattern_base(lo0, hi, j + 1), f2 = pattern_base(lo0, hi, j + 2),
                               f3 = pattern_base(lo0, hi, j + 3);
                if ((v.x ^ f0 ^ es_x) | (v.y ^ f1 ^ es_x) | (v.z ^ f2 ^ es_x) | (v.w ^ f3 ^ es_x)) {     // rare: a fault in this vector
                    mm.word(v.x, f0 ^ es_x, w0 + j);
                    mm.word(v.y, f1 ^ es_x, w0 + j + 1);
                    mm.word(v.z, f2 ^ es_x, w0 + j + 2);
                    mm.word(v.w, f3 ^ es_x, w0 + j + 3);
                }
                if (write) st[i] = make_uint4(f0 ^ ws_x, f1 ^ ws_x, f2 ^ ws_x, f3 ^ ws_x);
            }
            if (write) {
                fence_proxy_async_smem();          // generic-proxy writes of the stage -> visible to the bulk store
                __syncwarp();
                if (lane == 0) {
                    bulk_s2g(a.buf + chunk_off(k), ring + cs * kStageBytes, chunk_len(k), pol);
                    bulk_commit();
                    if (issued < n_my) {
                        bulk_wait_read<1>();       // the store of chunk k-1 has read its stage, which the next load reuses
                        load_next();
                    }
                }
            } else {
                __syncwarp();
                if (lane == 0 && issued < n_my) load_next();   // stage cs is free again: issued == k + kStages
            }
            advance();
        }
    }
    if (lane == 0) bulk_wait_all();

    // the <16-byte word tail that bulk copies cannot carry: one thread of the grid
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (uint64_t off = bulk_bytes; off < a.bytes; off += 4) {
            uint32_t* p = reinterpret_cast<uint32_t*>(a.buf + off);
            const uint64_t w = a.base_word + (off >> 2);
            if (verify) mm.word(*p, b200_pattern_word(w, a.expect_seed), w);
            if (write) *p = b200_pattern_word(w, a.write_seed);
        }
    }
    mm.publish(a.res);
}

int launch_element(int sms, uint8_t* buf, uint64_t bytes, uint64_t base_word, int flags, uint32_t es, uint32_t ws,
                   unsigned long long* d_res, cudaStream_t stream) {
    if (!bytes || !(flags & (B200PROBE_MEMTEST_VERIFY | B200PROBE_MEMTEST_WRITE))) return 0;
    const int smem = kWarps * kStages * kStageBytes;
    B200_CUDA_TRY(cudaFuncSetAttribute(hbm_memtest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    MemtestArgs a{buf, bytes, base_word, flags, es, ws, d_res};
    const uint64_t nchunks = ((bytes & ~15ull) + kStageBytes - 1) / kStageBytes;
    const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)sms, (nchunks + kWarps - 1) / kWarps));
    hbm_memtest_kernel<<<grid, kWarps * 32, smem, stream>>>(a);
    B200_CUDA_TRY(cudaGetLastError());
    return 0;
}

constexpr unsigned long long kResInit[3] = {0, ~0ull, 0};

// Reads the three device counters back (synchronising the stream) and resets them for the next element.
int take_results(unsigned long long* d_res, cudaStream_t stream, unsigned long long h[3]) {
    B200_CUDA_TRY(cudaMemcpyAsync(h, d_res, sizeof(kResInit), cudaMemcpyDeviceToHost, stream));
    B200_CUDA_TRY(cudaMemcpyAsync(d_res, kResInit, sizeof(kResInit), cudaMemcpyHostToDevice, stream));
    B200_CUDA_TRY(cudaStreamSynchronize(stream));
    return 0;
}

double now_ms() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}

// Everything the entry allocates; freed on every path by the destructor.
struct MemtestState {
    int ordinal = -1;
    std::vector<void*> chunks;
    std::vector<uint64_t> sizes;
    unsigned long long* d_res = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    ~MemtestState() {
        if (ordinal < 0) return;
        cudaSetDevice(ordinal);
        if (stream) cudaStreamSynchronize(stream);
        for (void* p : chunks) cudaFree(p);
        if (d_res) cudaFree(d_res);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (stream) cudaStreamDestroy(stream);
    }
};

int64_t delta(int64_t before, int64_t after) { return before < 0 || after < 0 ? -1 : after - before; }

}  // namespace

extern "C" {

int b200probe_memtest_element(int ordinal, void* buf, uint64_t bytes, uint64_t base_word, int flags, uint32_t expect_seed, uint32_t write_seed,
                              uint64_t* bad_words, uint64_t* first_bad_word, uint32_t* bad_bits) {
    if (bytes & 3) { b200::set_error("bytes=%llu is not a multiple of 4", (unsigned long long)bytes); return B200PROBE_EINVAL; }
    if ((uintptr_t)buf & 15) { b200::set_error("buffer must be 16-byte aligned"); return B200PROBE_EINVAL; }
    if (flags & ~(B200PROBE_MEMTEST_VERIFY | B200PROBE_MEMTEST_WRITE)) { b200::set_error("unknown memtest flags %d", flags); return B200PROBE_EINVAL; }
    b200::DevProps props;
    int rc = b200::device_props(ordinal, &props);
    if (rc) return rc;
    B200_CUDA_TRY(cudaSetDevice(ordinal));
    // The per-thread default stream is ordered after the caller's work on the legacy default stream (a buffer the caller
    // just wrote), and the stream-ordered allocation of the three counters costs no device-wide synchronisation.
    const cudaStream_t st = cudaStreamPerThread;
    unsigned long long* d_res = nullptr;
    B200_ALLOC_TRY(cudaMallocAsync((void**)&d_res, sizeof(kResInit), st));
    unsigned long long h[3];
    const cudaError_t e = cudaMemcpyAsync(d_res, kResInit, sizeof(kResInit), cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) { b200::set_error("cudaMemcpyAsync: %s", cudaGetErrorString(e)); rc = b200::cuda_rc((int)e); }
    if (!rc) rc = launch_element(props.sms, (uint8_t*)buf, bytes, base_word, flags, expect_seed, write_seed, d_res, st);
    if (!rc) rc = take_results(d_res, st, h);
    cudaFreeAsync(d_res, st);
    B200_CUDA_TRY(cudaStreamSynchronize(st));
    if (rc) return rc;
    if (bad_words) *bad_words = h[0];
    if (first_bad_word) *first_bad_word = h[1];
    if (bad_bits) *bad_bits = (uint32_t)h[2];
    return 0;
}

int b200probe_hbm_memtest(int idx, const b200probe_memtest_cfg_t* cfg_in, b200probe_memtest_result_t* out) {
    if (!out) return B200PROBE_EINVAL;
    memset(out, 0, sizeof(*out));
    out->first_bad_word = ~0ull;
    out->first_bad_element = -1;
    out->ecc_corrected_delta = out->ecc_uncorrected_delta = -1;
    b200probe_memtest_cfg_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    if (cfg_in) cfg = *cfg_in;
    if (cfg.fraction == 0) cfg.fraction = 0.9;
    if (!cfg.chunk_bytes) cfg.chunk_bytes = 1ull << 30;
    if (cfg.passes <= 0) cfg.passes = 1;
    if (!cfg.seed) cfg.seed = 0xB200u;
    if (!(cfg.fraction > 0 && cfg.fraction <= 1) || (cfg.chunk_bytes & 4095)) {
        b200::set_error("memtest: fraction must be in (0, 1] and chunk_bytes a multiple of 4096");
        return B200PROBE_EINVAL;
    }
    int ordinal = -1;
    int rc = b200::cuda_ordinal_of(idx, &ordinal);
    if (rc) return rc;
    b200::DevProps props;
    rc = b200::device_props(ordinal, &props);
    if (rc) return rc;

    b200probe_ecc_status_t ecc0;
    rc = b200probe_hbm_ecc(idx, &ecc0);
    if (rc) return rc;
    B200_CUDA_TRY(cudaSetDevice(ordinal));
    MemtestState s;
    s.ordinal = ordinal;
    // the small things first: once the chunks hold the free memory there may be none left for them
    B200_CUDA_TRY(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    B200_CUDA_TRY(cudaEventCreate(&s.e0));
    B200_CUDA_TRY(cudaEventCreate(&s.e1));
    B200_ALLOC_TRY(cudaMalloc(&s.d_res, sizeof(kResInit)));
    B200_CUDA_TRY(cudaMemcpyAsync(s.d_res, kResInit, sizeof(kResInit), cudaMemcpyHostToDevice, s.stream));
    size_t free_b = 0, total_b = 0;
    B200_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    out->free_before = free_b;
    out->total = total_b;

    uint64_t target = (uint64_t)(cfg.fraction * (double)free_b) & ~4095ull;
    if (cfg.max_bytes) target = std::min<uint64_t>(target, cfg.max_bytes & ~4095ull);
    const double t_alloc = now_ms();
    uint64_t got = 0;
    while (got < target) {
        const uint64_t want = std::min(cfg.chunk_bytes, target - got);
        void* p = nullptr;
        const cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); break; }     // a tenant took the rest: test what we hold
        B200_CUDA_TRY(e);
        s.chunks.push_back(p);
        s.sizes.push_back(want);
        got += want;
    }
    out->alloc_ms = now_ms() - t_alloc;
    out->chunks = (int)s.chunks.size();
    if (got == 0 || got < cfg.min_bytes) {
        b200::set_error("memtest: allocated %llu of the %llu bytes needed (free %zu)", (unsigned long long)got,
                        (unsigned long long)std::max<uint64_t>(cfg.min_bytes, 1), free_b);
        return B200PROBE_ENOMEM;
    }

    struct Element { int flags; uint32_t es, ws; };
    const uint32_t s0 = cfg.seed, s1 = cfg.seed ^ kSeed1Xor;
    const Element march[4] = {
        {B200PROBE_MEMTEST_WRITE, 0, s0},
        {B200PROBE_MEMTEST_VERIFY | B200PROBE_MEMTEST_WRITE, s0, ~s0},
        {B200PROBE_MEMTEST_VERIFY | B200PROBE_MEMTEST_WRITE, ~s0, s1},
        {B200PROBE_MEMTEST_VERIFY, s1, 0},
    };
    B200_CUDA_TRY(cudaEventRecord(s.e0, s.stream));
    for (int pass = 0; pass < cfg.passes; ++pass) {
        for (int el = 0; el < 4; ++el) {
            uint64_t base_word = 0;
            for (size_t c = 0; c < s.chunks.size(); ++c) {
                rc = launch_element(props.sms, (uint8_t*)s.chunks[c], s.sizes[c], base_word, march[el].flags, march[el].es, march[el].ws,
                                    s.d_res, s.stream);
                if (rc) return rc;
                base_word += s.sizes[c] >> 2;
            }
            if (!(march[el].flags & B200PROBE_MEMTEST_VERIFY)) continue;
            unsigned long long h[3];
            rc = take_results(s.d_res, s.stream, h);
            if (rc) return rc;
            if (h[0]) {
                out->bad_words += h[0];
                out->bad_bits |= (uint32_t)h[2];
                if (out->first_bad_element < 0) { out->first_bad_element = el; out->first_bad_word = h[1]; }
            }
        }
    }
    B200_CUDA_TRY(cudaEventRecord(s.e1, s.stream));
    B200_CUDA_TRY(cudaEventSynchronize(s.e1));
    float ms = 0;
    B200_CUDA_TRY(cudaEventElapsedTime(&ms, s.e0, s.e1));
    out->bytes_tested = got;
    out->passes = cfg.passes;
    out->test_ms = ms;
    out->gbs = ms > 0 ? 6.0 * (double)got * cfg.passes / (ms * 1e-3) / 1e9 : 0.0;

    rc = b200probe_hbm_ecc(idx, &out->ecc_after);
    if (rc) return rc;
    out->ecc_corrected_delta = delta(ecc0.corrected_volatile, out->ecc_after.corrected_volatile);
    out->ecc_uncorrected_delta = delta(ecc0.uncorrected_volatile, out->ecc_after.uncorrected_volatile);
    return 0;
}

}  // extern "C"
