// tcgen05 tensor-core GEMM probe for sm_100a (SURVEY.md §8a row a13; no reference counterpart).
//
//   C[M][N] (bf16) = A[M][K] (bf16, K-major) * B[N][K]^T (bf16, K-major), fp32 accumulate in TMEM.
//
// Persistent, warp-specialised, one CTA per SM:
//   warp 0   TMA producer   cp.async.bulk.tensor (SASS UTMALDG) 128B-swizzled A/B tiles -> smem ring
//   warp 1   MMA issuer     one lane issues tcgen05.mma (SASS UTCHMMA) M=128 N=256 K=16, smem x smem -> TMEM
//   warp 2   TMEM allocator tcgen05.alloc 512 columns = two 128x256 fp32 accumulators (double buffer)
//   warps 4-7 epilogue      tcgen05.ld (LDTM) 32 lanes x 32 columns, two register sets in flight -> cvt bf16 ->
//                           128B-swizzled shared-memory staging -> cp.async.bulk.tensor store (SASS UTMASTG), 64 columns at a time
// Pipelines: smem full/empty mbarriers (TMA <-> MMA), TMEM full/empty mbarriers (MMA <-> epilogue),
// so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// Roofline: tensor bound.  Algorithmic work per launch: 2*M*N*K flop.
// Two operand classes (cfg.operands):
//   0 EXACT    closed-form values k/128 (k integer): every partial sum is exactly representable in fp32, so C is
//              bit-exact against the fp64 oracle after one bf16 RNE (the probe's default: a health verdict with no tolerance)
//   1 UNIFORM  SURVEY.md §8d's input class: bf16 U(-1,1) from Philox4x32-10, key (seed, 0); sampled outputs against fp64
//              dot products within |err| <= 2^-8 |ref| + 2^-10 sqrt(K) (final bf16 rounding + fp32 accumulation allowance)
// FP8: gemm_e4m3_tn_2cta_512_kernel is the 512 x 256 kernel's body with E4M3 operands (tcgen05.mma kind::f8f6f4, SASS UTCQMMA,
// K=32 per MMA, 128 elements = the same 128 bytes per k-block) and the same two operand classes in E4M3 (DESIGN.md §4.5).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <pthread.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "common.h"

namespace {

constexpr int BM = 128, BN = 256, BK = 64, UMMA_K = 16;
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = BM * BK * 2;          // 16 KiB
constexpr int B_STAGE_BYTES = BN * BK * 2;          // 32 KiB
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int NUM_THREADS = 256;
constexpr int TMEM_COLS = 512;
constexpr int GROUP_M = 16;                         // rasterisation: 16 m-tiles per band (L2 reuse)
constexpr int EPI_UNIT_COLS = 64;                   // one TMA store = 32 rows x 64 bf16 columns = 32 x 128 B (one swizzle atom wide)
constexpr int EPI_BUF_BYTES = 32 * EPI_UNIT_COLS * 2;                 // 4 KiB
constexpr int EPI_BYTES = 4 /*warps*/ * 2 /*buffers*/ * EPI_BUF_BYTES;    // 32 KiB
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + 1024 /*align*/ + 256 /*barriers*/;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst_smem),
                 "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// all previously issued MMAs of this thread arrive on the mbarrier when they complete
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
          "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
          "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src_smem, int c0, int c1, uint64_t pol = 0) {
    if (pol)
        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"((uint64_t)map), "r"(src_smem), "r"(c0),
                     "r"(c1), "l"(pol)
                     : "memory");
    else
        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"((uint64_t)map), "r"(src_smem), "r"(c0), "r"(c1)
                     : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 32 fp32 accumulator columns of this lane's row -> 32 bf16 -> the 64-byte half `half` of the row's 128-byte line in the
// staging buffer, in the SWIZZLE_128B layout the C tensor map expects: 16-byte chunk j of row r sits at chunk j ^ (r & 7).
// (Rows are 128 B apart, so the 8 lanes of a store phase hit 8 different chunk columns: conflict-free.)
__device__ __forceinline__ void pack_half_row(const uint32_t (&v)[32], uint8_t* row, int half, int lane) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t pk[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 2 * i]), __uint_as_float(v[8 * j + 2 * i + 1]));
            pk[i] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(row + (((half * 4 + j) ^ (lane & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}

// Epilogue of one 32-row x 256-column slice (this warp's TMEM lane quadrant of one accumulator).  tcgen05.ld of the next 32
// columns is in flight while the previous 32 are converted (two register sets); 64 columns at a time leave through a
// swizzled staging buffer and ONE tensor store (full 128-byte lines instead of 16-byte pieces of 32 different lines);
// two staging buffers per warp, so a store drains while the next unit is packed.  `release` hands the accumulator back
// to the MMA issuer as soon as the last tcgen05.ld has landed, before the stores finish.
template <class Release>
__device__ __forceinline__ void epilogue_slice(uint32_t taddr, uint8_t* stage, uint32_t& ubuf, const CUtensorMap* tmc, int row0, int col0, int lane,
                                               Release release, uint64_t polc = 0) {
    uint32_t va[32], vb[32];
    tmem_ld_32x32(taddr, va);
    tmem_ld_wait();
#pragma unroll
    for (int u = 0; u < BN / EPI_UNIT_COLS; ++u) {
        tmem_ld_32x32(taddr + u * EPI_UNIT_COLS + 32, vb);          // in flight during the conversion of va
        if (lane == 0) bulk_wait_read1();                           // the store that read this buffer two units ago is done with it
        __syncwarp();
        uint8_t* buf = stage + ubuf * EPI_BUF_BYTES;
        pack_half_row(va, buf + lane * 128, 0, lane);
        tmem_ld_wait();
        if (u + 1 < BN / EPI_UNIT_COLS) tmem_ld_32x32(taddr + (u + 1) * EPI_UNIT_COLS, va);
        else release();                                             // every column of this accumulator slice is in registers
        pack_half_row(vb, buf + lane * 128, 1, lane);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
            tma_store_2d(tmc, smem_u32(buf), col0 + u * EPI_UNIT_COLS, row0, polc);
            bulk_commit_group();
        }
        ubuf ^= 1;
        if (u + 1 < BN / EPI_UNIT_COLS) tmem_ld_wait();
    }
}

// K-major operand tile [rows][64 bf16] written by TMA with SWIZZLE_128B: 8-row x 128-byte atoms,
// 1024 bytes apart (SBO); LBO is unused for swizzled K-major layouts; descriptor version 1 (sm_100).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;                     // leading byte offset (ignored)
    d |= (uint64_t)(1024 >> 4) << 32;           // stride byte offset
    d |= (uint64_t)1 << 46;                     // version
    d |= (uint64_t)2 << 61;                     // SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

struct TileCoord { int m0, n0; };
__device__ __forceinline__ TileCoord tile_coord(int t, int num_m, int num_n) {
    const int per_band = GROUP_M * num_n;
    const int band = t / per_band;
    const int first_m = band * GROUP_M;
    const int rows = min(GROUP_M, num_m - first_m);
    const int in_band = t - band * per_band;
    return {(first_m + in_band % rows) * BM, (in_band / rows) * BN};
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const __grid_constant__ CUtensorMap tma_c,
                    int M, int N, int K) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + STAGES * A_STAGE_BYTES;
    uint8_t* smem_epi = smem + STAGES * STAGE_BYTES;            // 4 warps x 2 x 4 KiB, 1024-aligned (swizzle atoms)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_epi + EPI_BYTES);
    uint64_t* full = bars;                  // [STAGES]
    uint64_t* empty = bars + STAGES;        // [STAGES]
    uint64_t* tfull = bars + 2 * STAGES;    // [2]
    uint64_t* tempty = tfull + 2;           // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_m = M / BM, num_n = N / BN, num_tiles = num_m * num_n, num_kb = K / BK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_b) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_c) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&full[s]), 1); mbar_init(smem_u32(&empty[s]), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(smem_u32(&tfull[a]), 1); mbar_init(smem_u32(&tempty[a]), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {                                   // ===== TMA producer =====
            uint32_t stage = 0, phase = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
                const TileCoord tc = tile_coord(t, num_m, num_n);
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(smem_u32(&empty[stage]), phase ^ 1);
                    const uint32_t fb = smem_u32(&full[stage]);
                    mbar_expect_tx(fb, STAGE_BYTES);
                    tma_load_2d(smem_u32(smem_a + stage * A_STAGE_BYTES), &tma_a, fb, kb * BK, tc.m0);
                    tma_load_2d(smem_u32(smem_b + stage * B_STAGE_BYTES), &tma_b, fb, kb * BK, tc.n0);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {                                   // ===== MMA issuer =====
            uint32_t stage = 0, phase = 0, it = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
                const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
                mbar_wait(smem_u32(&tempty[acc]), acc_phase ^ 1);      // epilogue drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(smem_u32(&full[stage]), phase);          // TMA bytes landed
                    tc_fence_after();
                    const uint64_t a_desc = make_smem_desc(smem_u32(smem_a + stage * A_STAGE_BYTES));
                    const uint64_t b_desc = make_smem_desc(smem_u32(smem_b + stage * B_STAGE_BYTES));
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        // +32 bytes per K=16 step inside the 128-byte swizzle atom (address field is >>4)
                        umma_bf16(d_tmem, a_desc + (uint64_t)(k * 2), b_desc + (uint64_t)(k * 2), kIdesc, (kb | k) != 0);
                    }
                    umma_commit(smem_u32(&empty[stage]));              // smem slot free when these MMAs retire
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(smem_u32(&tfull[acc]));                    // accumulator ready for the epilogue
            }
        }
    } else if (warp >= 4) {                                // ===== epilogue =====
        const int q = warp - 4;                            // == warp % 4: the TMEM lane quadrant this warp may read
        uint32_t it = 0, ubuf = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const TileCoord tc = tile_coord(t, num_m, num_n);
            const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
            mbar_wait(smem_u32(&tfull[acc]), acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
            const uint32_t tempty_bar = smem_u32(&tempty[acc]);
            epilogue_slice(taddr, smem_epi + q * 2 * EPI_BUF_BYTES, ubuf, &tma_c, tc.m0 + q * 32, tc.n0, lane, [&]() {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar);
            });
        }
        if (lane == 0) bulk_wait_all0();                   // the staging buffers are read by the TMA unit until then
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

// ---- cta_group::2 (CTA pair) forms -------------------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;     // shared::cluster address of the same offset in the even (leader) CTA
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// both CTAs of the pair issue their loads; the bytes complete on the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst_smem, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst_smem),
                 "l"((uint64_t)map), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the mbarrier at this offset in BOTH CTAs of the pair when the issued MMAs retire
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar & kPeerBitMask) : "memory");
}
// tuning knobs of the CTA-pair kernel (environment, experiments only; defaults = the shipped schedule)
struct GemmTune {
    int group_m;            // m-tiles (of 256 rows) per rasterisation band
    int pol_a, pol_b;       // L2 eviction policy of the A / B tensor loads: 0 none, 1 evict_first, 2 evict_last
    int pol_c;              // ... and of the C tensor stores
    int prefetch;           // 512 x 256 kernel: k-blocks by which an L2 prefetch of the operand boxes runs ahead of the loads (0 = none)
    int expt;               // attribution experiments (WRONG results): 1 = the epilogue hands the accumulators back without reading them
    int epi;                // 512 x 256 kernel epilogue: 0 = 32-byte stores from registers (default), 1 = staged tensor stores
    int skew;               // 512 x 256 kernel: k-blocks by which accumulator 1 runs behind accumulator 0 (0..3), see the MMA issuer
};
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* map, int c0, int c1) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"((uint64_t)map), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ uint64_t l2_policy(int kind) {
    uint64_t p = 0;
    if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    else if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tma_load_2d_2sm_hint(uint32_t dst_smem, const CUtensorMap* map, uint32_t bar, int c0, int c1, uint64_t pol) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst_smem),
                 "l"((uint64_t)map), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(pol)
                 : "memory");
}
constexpr int STAGES2 = 6;
constexpr int A2_STAGE_BYTES = BM * BK * 2;             // this CTA's 128 rows of the 256-row A tile
constexpr int B2_STAGE_BYTES = (BN / 2) * BK * 2;       // this CTA's 128 of the 256 B rows
constexpr int STAGE2_BYTES = A2_STAGE_BYTES + B2_STAGE_BYTES;     // 32 KiB per CTA per stage
constexpr int SMEM2_BYTES = STAGES2 * STAGE2_BYTES + EPI_BYTES + 1024 + 256;
static_assert(SMEM2_BYTES <= 232448 && SMEM_BYTES <= 232448, "227 KiB of shared memory per CTA");
constexpr uint32_t kIdesc2 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);   // M = 256

__device__ __forceinline__ TileCoord tile_coord2(int t, int num_m, int num_n, int group) {     // tiles of (2*BM) x BN, `group` m-tiles per band
    const int per_band = group * num_n;
    const int band = t / per_band;
    const int first_m = band * group;
    const int rows = min(group, num_m - first_m);
    const int in_band = t - band * per_band;
    return {(first_m + in_band % rows) * 2 * BM, (in_band / rows) * BN};
}

// C tile 256 x 256 per CTA PAIR: UMMA M=256 N=256 K=16 with cta_group::2.  Each CTA stages its own
// 128 A rows and 128 of the 256 B rows (half the shared-memory fill and L2 traffic per flop of the
// 1-CTA kernel), holds its 128 accumulator rows in its own TMEM and runs its own epilogue.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
gemm_bf16_tn_2cta_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const __grid_constant__ CUtensorMap tma_c,
                         int M, int N, int K, GemmTune tune) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + STAGES2 * A2_STAGE_BYTES;
    uint8_t* smem_epi = smem + STAGES2 * STAGE2_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_epi + EPI_BYTES);
    uint64_t* full = bars;                   // [STAGES2]  used in the leader only
    uint64_t* empty = bars + STAGES2;        // [STAGES2]  one per CTA, signalled by multicast commit
    uint64_t* tfull = bars + 2 * STAGES2;    // [2]        one per CTA, signalled by multicast commit
    uint64_t* tempty = tfull + 2;            // [2]        used in the leader only: 8 epilogue warps arrive
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();
    const bool leader = cta_rank == 0;
    const int num_m = M / (2 * BM), num_n = N / BN, num_tiles = num_m * num_n, num_kb = K / BK;
    const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_b) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tma_c) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES2; ++s) { mbar_init(smem_u32(&full[s]), 1); mbar_init(smem_u32(&empty[s]), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(smem_u32(&tfull[a]), 1); mbar_init(smem_u32(&tempty[a]), 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {                                   // ===== TMA producer (both CTAs) =====
            uint32_t stage = 0, phase = 0;
            const uint64_t pa = l2_policy(tune.pol_a), pb = l2_policy(tune.pol_b);
            for (int t = pair; t < num_tiles; t += num_pairs) {
                const TileCoord tc = tile_coord2(t, num_m, num_n, tune.group_m);
                const int my_m = tc.m0 + (int)cta_rank * BM, my_n = tc.n0 + (int)cta_rank * (BN / 2);
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(smem_u32(&empty[stage]), phase ^ 1);
                    const uint32_t fb = smem_u32(&full[stage]);
                    if (leader) mbar_expect_tx(fb, 2 * STAGE2_BYTES);      // both CTAs' bytes land on the leader's barrier
                    if (tune.pol_a) tma_load_2d_2sm_hint(smem_u32(smem_a + stage * A2_STAGE_BYTES), &tma_a, fb, kb * BK, my_m, pa);
                    else tma_load_2d_2sm(smem_u32(smem_a + stage * A2_STAGE_BYTES), &tma_a, fb, kb * BK, my_m);
                    if (tune.pol_b) tma_load_2d_2sm_hint(smem_u32(smem_b + stage * B2_STAGE_BYTES), &tma_b, fb, kb * BK, my_n, pb);
                    else tma_load_2d_2sm(smem_u32(smem_b + stage * B2_STAGE_BYTES), &tma_b, fb, kb * BK, my_n);
                    if (++stage == STAGES2) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (leader && lane == 0) {                         // ===== MMA issuer (leader CTA only) =====
            uint32_t stage = 0, phase = 0, it = 0;
            for (int t = pair; t < num_tiles; t += num_pairs, ++it) {
                const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
                mbar_wait(smem_u32(&tempty[acc]), acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(smem_u32(&full[stage]), phase);
                    tc_fence_after();
                    const uint64_t a_desc = make_smem_desc(smem_u32(smem_a + stage * A2_STAGE_BYTES));
                    const uint64_t b_desc = make_smem_desc(smem_u32(smem_b + stage * B2_STAGE_BYTES));
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k)
                        umma_bf16_2sm(d_tmem, a_desc + (uint64_t)(k * 2), b_desc + (uint64_t)(k * 2), kIdesc2, (kb | k) != 0);
                    umma_commit_2sm(smem_u32(&empty[stage]));
                    if (++stage == STAGES2) { stage = 0; phase ^= 1; }
                }
                umma_commit_2sm(smem_u32(&tfull[acc]));
            }
        }
    } else if (warp >= 4) {                                // ===== epilogue (both CTAs, own 128 rows) =====
        const int q = warp - 4;
        uint32_t it = 0, ubuf = 0;
        const uint64_t polc = l2_policy(tune.pol_c);
        for (int t = pair; t < num_tiles; t += num_pairs, ++it) {
            const TileCoord tc = tile_coord2(t, num_m, num_n, tune.group_m);
            const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
            mbar_wait(smem_u32(&tfull[acc]), acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
            const uint32_t tempty_bar = smem_u32(&tempty[acc]);
            epilogue_slice(taddr, smem_epi + q * 2 * EPI_BUF_BYTES, ubuf, &tma_c, tc.m0 + (int)cta_rank * BM + q * 32, tc.n0, lane, [&]() {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(tempty_bar);
            }, polc);
        }
        if (lane == 0) bulk_wait_all0();
    }
    tc_fence_before();
    cluster_sync_all();            // the peer's MMAs read this CTA's shared memory: nobody leaves early
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

// ---- epilogue in 32-column units (the 512 x 256 kernel: EIGHT epilogue warps, one 32-row x 256-column accumulator slice each) ----
// One unit = one tcgen05.ld (32 lanes x 32 fp32 columns) -> 32 bf16 = a 64-byte row segment -> staging buffer in the SWIZZLE_64B
// layout of the 32-column C map (16-byte chunk j of row r at chunk j ^ ((r >> 1) & 3): rows 64 B apart, conflict-free) -> one
// tensor store of 32 rows x 64 B.  Two register sets and two 2 KiB buffers per warp: the next load and the previous store are in
// flight while a unit is converted.  8 warps x 2 x 2 KiB = the same 32 KiB the 64-column path uses for 4 warps.
constexpr int EPI32_BUF_BYTES = 32 * 32 * 2;      // 2 KiB
__device__ __forceinline__ void pack_row32(const uint32_t (&v)[32], uint8_t* row, int lane) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t pk[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 2 * i]), __uint_as_float(v[8 * j + 2 * i + 1]));
            pk[i] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(row + ((j ^ ((lane >> 1) & 3)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}
template <class Release>
__device__ __forceinline__ void epilogue_slice32(uint32_t taddr, uint8_t* stage, uint32_t& ubuf, const CUtensorMap* tmc32, int row0, int col0, int lane,
                                                 Release release, uint64_t polc) {
    uint32_t va[32], vb[32];
    tmem_ld_32x32(taddr, va);
    tmem_ld_wait();
#pragma unroll
    for (int u = 0; u < BN / 32; u += 2) {
        // unit u from va while the load of unit u+1 is in flight
        tmem_ld_32x32(taddr + (u + 1) * 32, vb);
        if (lane == 0) bulk_wait_read1();
        __syncwarp();
        uint8_t* buf = stage + ubuf * EPI32_BUF_BYTES;
        pack_row32(va, buf + lane * 64, lane);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) { tma_store_2d(tmc32, smem_u32(buf), col0 + u * 32, row0, polc); bulk_commit_group(); }
        ubuf ^= 1;
        tmem_ld_wait();
        // unit u+1 from vb while the load of unit u+2 is in flight
        if (u + 2 < BN / 32) tmem_ld_32x32(taddr + (u + 2) * 32, va);
        else release();                                             // the whole slice is in registers
        if (lane == 0) bulk_wait_read1();
        __syncwarp();
        buf = stage + ubuf * EPI32_BUF_BYTES;
        pack_row32(vb, buf + lane * 64, lane);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) { tma_store_2d(tmc32, smem_u32(buf), col0 + (u + 1) * 32, row0, polc); bulk_commit_group(); }
        ubuf ^= 1;
        if (u + 2 < BN / 32) tmem_ld_wait();
    }
}

// ---- epilogue straight from registers: 32 fp32 columns -> 32 bf16 = 64 bytes of one C row = TWO 32-byte stores per lane
// (st.global.v8.b32, SASS STG.E.256: every store fills one whole 32-byte sector).  No staging buffer, no tensor store: at a tile
// boundary the TMA unit is busy prefetching the next tile's four operand stages (192 KiB per CTA), and small tensor stores queued
// behind those loads held the accumulators for about 3 us per tile (3.4 % of the step, measured by handing the accumulators back
// unread: tools/gemm_tune.py expt 1); plain stores go through the LSU and retire independently.
__device__ __forceinline__ void store_row32(const uint32_t (&v)[32], __nv_bfloat16* dst) {
    uint32_t pk[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
        pk[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]), "r"(pk[4]), "r"(pk[5]),
                 "r"(pk[6]), "r"(pk[7])
                 : "memory");
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + 16), "r"(pk[8]), "r"(pk[9]), "r"(pk[10]), "r"(pk[11]), "r"(pk[12]),
                 "r"(pk[13]), "r"(pk[14]), "r"(pk[15])
                 : "memory");
}
template <class Release>
__device__ __forceinline__ void epilogue_slice_direct(uint32_t taddr, __nv_bfloat16* crow /* this lane's row, first column of the tile */, bool row_ok,
                                                      Release release) {
    uint32_t va[32], vb[32];
    tmem_ld_32x32(taddr, va);
    tmem_ld_wait();
#pragma unroll
    for (int u = 0; u < BN / 32; u += 2) {
        tmem_ld_32x32(taddr + (u + 1) * 32, vb);                    // in flight while va is converted and stored
        if (row_ok) store_row32(va, crow + u * 32);
        tmem_ld_wait();
        if (u + 2 < BN / 32) tmem_ld_32x32(taddr + (u + 2) * 32, va);
        else release();                                             // the whole slice has left TMEM
        if (row_ok) store_row32(vb, crow + (u + 1) * 32);
        if (u + 2 < BN / 32) tmem_ld_wait();
    }
}

// ---- 512 x 256 per CTA pair ---------------------------------------------------------------------------------------------
// Each CTA of the pair stages 256 A rows (two 128-row halves) and 128 of the 256 B rows per k-block, and every k16 step issues
// TWO cta_group::2 MMAs (M256 N256 K16) against the same B stage: half h of both CTAs' A -> accumulator h (TMEM columns
// [256h, 256h+256)).  Per flop the shared-memory fill (and the L2 -> SM traffic behind it) is 3/4 of the 256 x 256 pair tile's:
// 768 operand rows per 512 x 256 x 64 block instead of 512 per 256 x 256 x 64.  At the 1 kW power cap that is what decides the
// clock: ncu had the 256 x 256 kernel at 47.9 % L2 throughput and 1.39 GHz next to cuBLAS's 512 x 256 kernel
// (nvjet_tst_256x256_64x4_2x1_2cta) at 30.3 % and 1.48 GHz on the same operands (profiles/ncu_gemm_vs_cublas_r02.txt).
// Price: both accumulators = all 512 TMEM columns, so a tile's epilogue is not hidden behind the next tile's MMAs; the kernel
// stays persistent, so the next tile's TMA prologue (4 stages) does run under the epilogue.
constexpr int STAGES3 = 4;
constexpr int A3_STAGE_BYTES = 2 * BM * BK * 2;         // this CTA's 256 A rows: 32 KiB, rows [128, 256) start 16 KiB in
constexpr int B3_STAGE_BYTES = (BN / 2) * BK * 2;       // this CTA's 128 of the 256 B rows: 16 KiB
constexpr int STAGE3_BYTES = A3_STAGE_BYTES + B3_STAGE_BYTES;
constexpr int SMEM3_BYTES = STAGES3 * STAGE3_BYTES + EPI_BYTES + 1024 + 256;
static_assert(SMEM3_BYTES <= 232448, "227 KiB of shared memory per CTA");

__device__ __forceinline__ TileCoord tile_coord3(int t, int num_m, int num_n, int group) {     // tiles of (4*BM) x BN
    const int per_band = group * num_n;
    const int band = t / per_band;
    const int first_m = band * group;
    const int rows = min(group, num_m - first_m);
    const int in_band = t - band * per_band;
    return {(first_m + in_band % rows) * 4 * BM, (in_band / rows) * BN};
}

// Operand kinds of the 512 x 256 kernel.  Every k-block is 128 bytes of each operand row (one SWIZZLE_128B atom) and four
// MMAs 32 bytes apart, so stage sizes, expect_tx counts, shared-memory descriptors and the epilogue are the same for both;
// the kind differs in the MMA, its instruction descriptor and the elements per k-block (the TMA K coordinate).
__device__ __forceinline__ void umma_e4m3_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
struct OperandBf16 {                                    // kind::f16, M256 N256 K16: 64 bf16 per k-block
    static constexpr int kKbElems = BK;
    static constexpr bool kE4m3 = false;
    static constexpr bool kStagedEpilogue = true;       // has a C tensor map (B200PROBE_GEMM_EPI=1)
};
struct OperandE4m3 {                                    // kind::f8f6f4, M256 N256 K32: 128 E4M3 per k-block
    static constexpr int kKbElems = 128;
    static constexpr bool kE4m3 = true;
    static constexpr bool kStagedEpilogue = false;
    // kind::f8f6f4 instruction descriptor: D = F32 (bit 4), A and B format E4M3 (0 in [7,10) and [10,13)), no negation, both
    // K-major (bits 15, 16 clear), N>>3 at [17,23), M>>4 at [24,29)
    static constexpr uint32_t kIdesc = (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);
};
static_assert(OperandE4m3::kKbElems * 1 == BK * 2, "an E4M3 k-block is the same 128 bytes as a bf16 one");
constexpr GemmTune kShippedTune3{4, 0, 0, 0, 0, 0, 0, 0};   // the 512 x 256 kernel's schedule with every knob at its default

constexpr int NUM_THREADS3 = 384;                       // warps 0-3: TMA producer, MMA issuer, TMEM allocator, idle; warps 4-11: epilogue
template <class Op>
__device__ __forceinline__ void gemm_tn_2cta_512(const CUtensorMap* tma_a, const CUtensorMap* tma_b, const CUtensorMap* tma_c,
                                                 __nv_bfloat16* __restrict__ C, int M, int N, int K, GemmTune tune) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + STAGES3 * A3_STAGE_BYTES;
    uint8_t* smem_epi = smem + STAGES3 * STAGE3_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_epi + EPI_BYTES);
    uint64_t* full = bars;                   // [STAGES3]  used in the leader only
    uint64_t* empty = bars + STAGES3;        // [STAGES3]  one per CTA, signalled by multicast commit
    uint64_t* tfull = bars + 2 * STAGES3;    // [2] one per accumulator and CTA, signalled by multicast commit: accumulator h of the tile is complete
    uint64_t* tempty = tfull + 2;            // [2] leader only: the 4 + 4 epilogue warps of accumulator h have it in registers
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();
    const bool leader = cta_rank == 0;
    // rows past M are zero-filled by the tensor loads and clipped by the tensor stores: any M that is a multiple of 128 works
    const int num_m = (M + 4 * BM - 1) / (4 * BM), num_n = N / BN, num_tiles = num_m * num_n, num_kb = K / Op::kKbElems;
    // cluster i sits on SMs 2(i-3), 2(i-3)+1 (tools/smid_probe.cu): consecutive pairs are neighbours on the chip already
    const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)tma_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)tma_b) : "memory");
        if constexpr (Op::kStagedEpilogue) asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)tma_c) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES3; ++s) { mbar_init(smem_u32(&full[s]), 1); mbar_init(smem_u32(&empty[s]), 1); }
        for (int h = 0; h < 2; ++h) { mbar_init(smem_u32(&tfull[h]), 1); mbar_init(smem_u32(&tempty[h]), 8); }    // 4 warps per accumulator in each CTA
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {                                   // ===== TMA producer (both CTAs) =====
            uint32_t stage = 0, phase = 0;
            const uint64_t pa = l2_policy(tune.pol_a), pb = l2_policy(tune.pol_b);
            // L2 prefetch `tune.prefetch` k-blocks ahead of the loads (across tile boundaries): about a quarter of the operand sectors
            // miss L2, and with 48 KiB per stage nearly every stage holds a miss, so without it a stage's latency is DRAM's
            auto prefetch_block = [&](long long gkb) {
                const int ti = pair + (int)(gkb / num_kb) * num_pairs;
                if (ti >= num_tiles) return;
                const TileCoord pc = tile_coord3(ti, num_m, num_n, tune.group_m);
                const int k0 = (int)(gkb % num_kb) * Op::kKbElems;
                tma_prefetch_l2_2d(tma_a, k0, pc.m0 + (int)cta_rank * 2 * BM);
                tma_prefetch_l2_2d(tma_b, k0, pc.n0 + (int)cta_rank * (BN / 2));
            };
            long long gkb = 0;
            for (int pf = 0; pf < tune.prefetch; ++pf) prefetch_block(pf);
            for (int t = pair; t < num_tiles; t += num_pairs) {
                const TileCoord tc = tile_coord3(t, num_m, num_n, tune.group_m);
                const int my_m = tc.m0 + (int)cta_rank * 2 * BM, my_n = tc.n0 + (int)cta_rank * (BN / 2);
                for (int kb = 0; kb < num_kb; ++kb, ++gkb) {
                    if (tune.prefetch) prefetch_block(gkb + tune.prefetch);
                    mbar_wait(smem_u32(&empty[stage]), phase ^ 1);
                    const uint32_t fb = smem_u32(&full[stage]);
                    if (leader) mbar_expect_tx(fb, 2 * STAGE3_BYTES);      // both CTAs' bytes land on the leader's barrier
                    if (tune.pol_a) tma_load_2d_2sm_hint(smem_u32(smem_a + stage * A3_STAGE_BYTES), tma_a, fb, kb * Op::kKbElems, my_m, pa);
                    else tma_load_2d_2sm(smem_u32(smem_a + stage * A3_STAGE_BYTES), tma_a, fb, kb * Op::kKbElems, my_m);
                    if (tune.pol_b) tma_load_2d_2sm_hint(smem_u32(smem_b + stage * B3_STAGE_BYTES), tma_b, fb, kb * Op::kKbElems, my_n, pb);
                    else tma_load_2d_2sm(smem_u32(smem_b + stage * B3_STAGE_BYTES), tma_b, fb, kb * Op::kKbElems, my_n);
                    if (++stage == STAGES3) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (leader && lane == 0) {                         // ===== MMA issuer (leader CTA only) =====
            // Accumulator 1 runs `d` k-blocks behind accumulator 0.  Both accumulators fill TMEM, so a tile's epilogue cannot hide
            // behind the next tile's MMAs as a whole — but with the skew accumulator 0 completes d blocks early and is drained
            // (TMEM reads: 64 B/clk, 2048 clocks per accumulator) while the tensor pipe still works on accumulator 1's last d
            // blocks, and accumulator 1 is drained under the next tile's first d blocks of accumulator 0.  A stage is released
            // when accumulator 1 has consumed it, so the loads' lookahead shrinks from STAGES3 to STAGES3 - d blocks.
            //   per tile:  A  acc0 blocks [0, d)                 B  acc1 block kb-d, acc0 block kb  (kb in [d, num_kb))
            //              C  acc1 blocks [num_kb-d, num_kb)     tfull[0] after B, tfull[1] after C;  d = 0: the plain order
            // MEASURED (tools/gemm_tune.py, 8192^3, sustained): d = 0 1432, d = 1 1422, d = 2 1312, d = 3 943 TFLOP/s — with four 48 KiB
            // stages the lost lookahead costs more than the hidden drain gains, so the default is d = 0 (B200PROBE_GEMM_SKEW).
            const int d = max(0, min(tune.skew, min(num_kb - 1, STAGES3 - 1)));
            long long g0 = 0, g1 = 0;                          // k-blocks consumed so far by accumulator 0 / 1 (the stage ring index)
            auto issue = [&](long long g, int h, int kb) {
                const uint32_t stage = (uint32_t)(g % STAGES3);
                const uint64_t a_desc = make_smem_desc(smem_u32(smem_a + stage * A3_STAGE_BYTES)) + (uint64_t)(h * ((BM * BK * 2) >> 4));
                const uint64_t b_desc = make_smem_desc(smem_u32(smem_b + stage * B3_STAGE_BYTES));
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k)
                    if constexpr (Op::kE4m3) umma_e4m3_2sm(tmem_base + h * BN, a_desc + (uint64_t)(k * 2), b_desc + (uint64_t)(k * 2), Op::kIdesc, (kb | k) != 0);
                    else umma_bf16_2sm(tmem_base + h * BN, a_desc + (uint64_t)(k * 2), b_desc + (uint64_t)(k * 2), kIdesc2, (kb | k) != 0);
            };
            auto wait_full = [&](long long g) {
                mbar_wait(smem_u32(&full[g % STAGES3]), (uint32_t)((g / STAGES3) & 1));
                tc_fence_after();
            };
            uint32_t it = 0;
            for (int t = pair; t < num_tiles; t += num_pairs, ++it) {
                mbar_wait(smem_u32(&tempty[0]), (it & 1) ^ 1);             // accumulator 0 of the previous tile is in registers
                tc_fence_after();
                for (int kb = 0; kb < d; ++kb, ++g0) { wait_full(g0); issue(g0, 0, kb); }
                mbar_wait(smem_u32(&tempty[1]), (it & 1) ^ 1);
                tc_fence_after();
                for (int kb = d; kb < num_kb; ++kb, ++g0, ++g1) {
                    wait_full(g0);
                    issue(g1, 1, kb - d);
                    umma_commit_2sm(smem_u32(&empty[g1 % STAGES3]));       // both accumulators are done with that stage
                    issue(g0, 0, kb);
                }
                umma_commit_2sm(smem_u32(&tfull[0]));
                for (int kb = num_kb - d; kb < num_kb; ++kb, ++g1) {
                    issue(g1, 1, kb);
                    umma_commit_2sm(smem_u32(&empty[g1 % STAGES3]));
                }
                umma_commit_2sm(smem_u32(&tfull[1]));
            }
        }
    } else if (warp >= 4) {                                // ===== epilogue (both CTAs): warp -> accumulator h, TMEM lane quadrant q =====
        const int q = warp & 3, h = (warp - 4) >> 2;       // a warp may read TMEM lanes [32 (warp % 4), +32)
        uint32_t it = 0, ubuf = 0;
        const uint64_t polc = l2_policy(tune.pol_c);
        const uint32_t tempty_bar = smem_u32(&tempty[h]);
        uint8_t* const stage = smem_epi + (warp - 4) * 2 * EPI32_BUF_BYTES;
        for (int t = pair; t < num_tiles; t += num_pairs, ++it) {
            const TileCoord tc = tile_coord3(t, num_m, num_n, tune.group_m);
            mbar_wait(smem_u32(&tfull[h]), it & 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + h * BN;
            const int row0 = tc.m0 + (int)cta_rank * 2 * BM + h * BM + q * 32;
            auto release = [&]() {
                tc_fence_before();                         // this warp's slice is in registers: 8 such arrivals free accumulator h
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(tempty_bar);
            };
            if (tune.expt == 1) { release(); continue; }   // how much of the step is the exposed epilogue?  (results are not written)
            if (tune.epi == 0) {
                const int row = row0 + lane;
                epilogue_slice_direct(taddr, C + (size_t)row * N + tc.n0, row < M, release);
                continue;
            }
            epilogue_slice32(taddr, stage, ubuf, tma_c, row0, tc.n0, lane, [&]() {
                tc_fence_before();                         // this warp's slice is in registers: 8 such arrivals free accumulator h
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(tempty_bar);
            }, polc);
        }
        if (lane == 0) bulk_wait_all0();
    }
    tc_fence_before();
    cluster_sync_all();            // the peer's MMAs read this CTA's shared memory: nobody leaves early
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS3, 1)
gemm_bf16_tn_2cta_512_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const __grid_constant__ CUtensorMap tma_c,
                             __nv_bfloat16* __restrict__ C, int M, int N, int K, GemmTune tune) {
    gemm_tn_2cta_512<OperandBf16>(&tma_a, &tma_b, &tma_c, C, M, N, K, tune);
}
// A [M][K] and B [N][K] E4M3, C [M][N] bf16: the shipped schedule, no tuning knobs (epilogue straight from registers, no C map)
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS3, 1)
gemm_e4m3_tn_2cta_512_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, __nv_bfloat16* __restrict__ C, int M, int N,
                             int K) {
    gemm_tn_2cta_512<OperandE4m3>(&tma_a, &tma_b, nullptr, C, M, N, K, kShippedTune3);
}

// `which`: bit 0 = matrix (0 A, 1 B), bit 1 = operand class (0 EXACT k/128, 1 UNIFORM Philox U(-1,1))
__global__ void gemm_fill_kernel(uint16_t* dst, uint64_t elems, uint32_t seed, int which) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    if (which & 2) {
        // one Philox block = 4 consecutive elements = one 8-byte store (dst is 16-byte aligned, elems a multiple of 4 up to the tail)
        const uint64_t nblk = elems >> 2;
        for (uint64_t b = i; b < nblk; b += stride) {
            uint32_t r[4];
            b200_philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)(which & 1), 0u, seed, 0u, r);
            uint16_t h[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t u = __float_as_uint((float)(r[j] >> 8) * (1.0f / 8388608.0f) - 1.0f);
                h[j] = (uint16_t)((u + 0x7fffu + ((u >> 16) & 1u)) >> 16);
            }
            *reinterpret_cast<uint2*>(dst + 4 * b) = make_uint2((uint32_t)h[0] | ((uint32_t)h[1] << 16), (uint32_t)h[2] | ((uint32_t)h[3] << 16));
        }
        for (uint64_t e = (nblk << 2) + i; e < elems; e += stride) dst[e] = b200_gemm_uniform_bits(e, seed, which & 1);
    } else {
        for (; i < elems; i += stride) dst[i] = b200_gemm_elem_bits(i, seed, which);
    }
}

// E4M3 operands (b200probe_gemm_fill with bit 2 of `which` set): one byte per element, four elements (one Philox block of the
// UNIFORM class) per 4-byte store, rounded by the hardware conversion (the host twin is b200_e4m3_rne)
__device__ __forceinline__ uint32_t e4m3x4(float x0, float x1, float x2, float x3) {
    uint16_t lo, hi;
    asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(x1), "f"(x0));       // x0 -> the low byte
    asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(x3), "f"(x2));
    return (uint32_t)lo | ((uint32_t)hi << 16);
}
__global__ void gemm_fill_e4m3_kernel(uint8_t* dst, uint64_t elems, uint32_t seed, int which) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const int mat = which & 1, uniform = (which >> 1) & 1;
    const uint64_t nblk = elems >> 2;
    for (uint64_t b = i; b < nblk; b += stride) {
        float x[4];
        if (uniform) {
            uint32_t r[4];
            b200_philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)mat, 0u, seed, 0u, r);
#pragma unroll
            for (int j = 0; j < 4; ++j) x[j] = (float)(r[j] >> 8) * (1.0f / 8388608.0f) - 1.0f;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) x[j] = b200_gemm_e4m3_value(4 * b + j, seed, mat, 0);
        }
        *reinterpret_cast<uint32_t*>(dst + 4 * b) = e4m3x4(x[0], x[1], x[2], x[3]);
    }
    for (uint64_t e = (nblk << 2) + i; e < elems; e += stride) dst[e] = (uint8_t)e4m3x4(b200_gemm_e4m3_value(e, seed, mat, uniform), 0.f, 0.f, 0.f);
}

__global__ void gather_kernel(const uint16_t* c, const uint64_t* idx, uint16_t* out, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = c[idx[i]];
}

// ---- tensor maps (driver entry point fetched through the runtime: no link-time libcuda dependency) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encode(EncodeTiledFn* fn) {
    static EncodeTiledFn cached = nullptr;
    if (!cached) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
        if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !p) {
            b200::set_error("cuTensorMapEncodeTiled unavailable (%s)", cudaGetErrorString(e));
            return e != cudaSuccess ? b200::cuda_rc(e) : B200PROBE_ENOCUDA;
        }
        cached = (EncodeTiledFn)p;
    }
    *fn = cached;
    return 0;
}

// [rows][inner] row-major -> box {box_cols (inner), box_rows}, 128B swizzle.  Operands: inner = K; C: inner = N.
// bf16 (the default): box_cols = 64 is one 128-byte row; box_cols = 32 selects the 64-byte-swizzled map of the 32-column
// epilogue units.  E4M3 operands: CU_TENSOR_MAP_DATA_TYPE_UINT8, 1 byte, box_cols = 128.  The L2 promotion experiment
// (B200PROBE_GEMM_L2_PROMOTION) belongs to the bf16 kernels: other element types get the default 256 B.
int make_map(CUtensorMap* map, const void* base, int rows, int inner, int box_rows, int box_cols = BK,
             CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, int elem_bytes = 2) {
    EncodeTiledFn enc = nullptr;
    int rc = get_encode(&enc);
    if (rc) return rc;
    cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)inner * elem_bytes};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    static const int l2prom = [] { const char* e = getenv("B200PROBE_GEMM_L2_PROMOTION"); return e ? atoi(e) : 256; }();      // experiments: 0, 64, 128, 256
    const int l2 = dtype == CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 ? l2prom : 256;
    const CUtensorMapL2promotion prom = l2 == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE : l2 == 64 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                                      : l2 == 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
    CUresult r = enc(map, dtype, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     box_cols * elem_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, prom, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { b200::set_error("cuTensorMapEncodeTiled failed: CUresult %d", (int)r); return B200PROBE_CUDA_BASE + 1; }
    return 0;
}
static_assert(EPI_UNIT_COLS == BK, "the C map reuses the operands' 64-element (128-byte) box width");

int check_shape(int m, int n, int k) {
    if (m <= 0 || n <= 0 || k <= 0 || m % BM || n % BN || k % BK) {
        b200::set_error("gemm: m,n,k must be positive multiples of %d,%d,%d (got %d,%d,%d)", BM, BN, BK, m, n, k);
        return B200PROBE_EINVAL;
    }
    return 0;
}
// the E4M3 kernel: CTA pairs of 256 rows, k-blocks of 128 elements
int check_shape_fp8(int m, int n, int k) {
    if (m <= 0 || n <= 0 || k <= 0 || m % (2 * BM) || n % BN || k % OperandE4m3::kKbElems) {
        b200::set_error("gemm_fp8: m,n,k must be positive multiples of %d,%d,%d (got %d,%d,%d)", 2 * BM, BN, OperandE4m3::kKbElems, m, n, k);
        return B200PROBE_EINVAL;
    }
    return 0;
}

double median_f(std::vector<float> v) {
    std::sort(v.begin(), v.end());
    size_t n = v.size();
    return n & 1 ? v[n / 2] : 0.5 * (v[n / 2 - 1] + v[n / 2]);
}

float bf16_bits_to_float(uint16_t b) {
    uint32_t u = (uint32_t)b << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
}
uint16_t float_to_bf16_rne(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    uint32_t r = 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)((u + r) >> 16);
}
double e4m3_bits_to_double(uint8_t v) {
    const int e = (v >> 3) & 15, m = v & 7;
    if (e == 15 && m == 7) return NAN;
    const double mag = e ? ldexp(8 + m, e - 10) : ldexp(m, -9);      // (1 + m/8) 2^(e-7), subnormal m/8 2^-6
    return (v & 0x80) ? -mag : mag;
}

// Per-device resident arena (like hbm_sweep.cu's): operands stay filled between calls with the same shape, seed, operand
// class and element type — the daemon probes periodically, and 384 MiB of cudaMalloc + two fills cost more than the ten
// timed GEMMs.  Operand buffers are sized for bf16; E4M3 operands use the first half of them.
struct GemmArena {
    pthread_mutex_t mu = PTHREAD_MUTEX_INITIALIZER;
    void *a = nullptr, *b = nullptr, *c = nullptr, *idx = nullptr, *out = nullptr;
    unsigned long long* partials = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int m = 0, n = 0, k = 0, operands = -1, samples_cap = 0;
    int e4m3 = -1;                                          // element type of the filled operands: 0 bf16, 1 E4M3
    uint32_t seed = 0;
    bool filled = false;
};
GemmArena g_gemm[B200PROBE_MAX_DEVICES];

void gemm_arena_free(GemmArena& g) {
    if (g.a) cudaFree(g.a);
    if (g.b) cudaFree(g.b);
    if (g.c) cudaFree(g.c);
    if (g.idx) cudaFree(g.idx);
    if (g.out) cudaFree(g.out);
    if (g.partials) cudaFree(g.partials);
    if (g.e0) cudaEventDestroy(g.e0);
    if (g.e1) cudaEventDestroy(g.e1);
    if (g.stream) cudaStreamDestroy(g.stream);
    g.a = g.b = g.c = g.idx = g.out = nullptr;
    g.partials = nullptr; g.e0 = g.e1 = nullptr; g.stream = nullptr;
    g.m = g.n = g.k = 0; g.operands = -1; g.e4m3 = -1; g.samples_cap = 0; g.filled = false;
}



int gemm_arena_reserve(GemmArena& g, int M, int N, int K, int samples) {
    if (!g.stream) {
        B200_CUDA_TRY(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
        B200_CUDA_TRY(cudaEventCreate(&g.e0));
        B200_CUDA_TRY(cudaEventCreate(&g.e1));
        B200_ALLOC_TRY(cudaMalloc(&g.partials, 32));
    }
    if (M != g.m || N != g.n || K != g.k) {
        if (g.a) cudaFree(g.a);
        if (g.b) cudaFree(g.b);
        if (g.c) cudaFree(g.c);
        g.a = g.b = g.c = nullptr; g.m = g.n = g.k = 0; g.filled = false;
        B200_ALLOC_TRY(cudaMalloc(&g.a, (size_t)M * K * 2));
        B200_ALLOC_TRY(cudaMalloc(&g.b, (size_t)N * K * 2));
        B200_ALLOC_TRY(cudaMalloc(&g.c, (size_t)M * N * 2));
        g.m = M; g.n = N; g.k = K;
    }
    if (samples > g.samples_cap) {
        if (g.idx) cudaFree(g.idx);
        if (g.out) cudaFree(g.out);
        g.idx = g.out = nullptr; g.samples_cap = 0;
        B200_ALLOC_TRY(cudaMalloc(&g.idx, (size_t)samples * 8));
        B200_ALLOC_TRY(cudaMalloc(&g.out, (size_t)samples * 2));
        g.samples_cap = samples;
    }
    return 0;
}

struct GemmLock {
    GemmArena& g;
    explicit GemmLock(GemmArena& x) : g(x) { pthread_mutex_lock(&g.mu); }
    ~GemmLock() { pthread_mutex_unlock(&g.mu); }
};

}  // namespace

extern "C" {

int b200probe_gemm_fill(int ordinal, void* dst, uint64_t elems, uint32_t seed, int which, void* stream) {
    b200::DevProps props;
    int rc = b200::device_props(ordinal, &props);
    if (rc) return rc;
    if (!dst || which < 0 || which > 7 || (((uintptr_t)dst) & 15)) return B200PROBE_EINVAL;
    B200_CUDA_TRY(cudaSetDevice(ordinal));
    if (elems && (which & 4)) gemm_fill_e4m3_kernel<<<props.sms * 8, 256, 0, (cudaStream_t)stream>>>((uint8_t*)dst, elems, seed, which & 3);
    else if (elems) gemm_fill_kernel<<<props.sms * 8, 256, 0, (cudaStream_t)stream>>>((uint16_t*)dst, elems, seed, which);
    B200_CUDA_TRY(cudaGetLastError());
    return 0;
}

uint16_t b200probe_gemm_operand_bits(uint64_t elem, uint32_t seed, int which) {
    if (which & 4) return b200_e4m3_rne(b200_gemm_e4m3_value(elem, seed, which & 1, (which >> 1) & 1));
    return (which & 2) ? b200_gemm_uniform_bits(elem, seed, which & 1) : b200_gemm_elem_bits(elem, seed, which & 1);
}

// kernel variant: 3 = CTA-pair kernel, 512 x 256 per pair (default when M is a multiple of 256; rows past M are zero-filled /
// clipped by the tensor maps), 2 = CTA-pair kernel, 256 x 256 per pair with double-buffered accumulators, 1 = single-CTA kernel
// (any M that is a multiple of 128).  B200PROBE_GEMM_VARIANT overrides, read per launch (tuning / A-B comparison).
static int gemm_variant_for(int m) {
    const char* e = getenv("B200PROBE_GEMM_VARIANT");
    const int forced = e ? atoi(e) : 0;
    if (forced == 1 || m % (2 * BM) != 0) return 1;
    return forced == 2 ? 2 : 3;
}

int b200probe_gemm_launch(int ordinal, const void* a, const void* b, void* c, int m, int n, int k, void* stream) {
    b200::DevProps props;
    int rc = b200::device_props(ordinal, &props);
    if (rc) return rc;
    rc = check_shape(m, n, k);
    if (rc) return rc;
    if (!a || !b || !c || (((uintptr_t)a | (uintptr_t)b | (uintptr_t)c) & 15)) { b200::set_error("gemm: operands must be 16-byte aligned device pointers"); return B200PROBE_EINVAL; }
    B200_CUDA_TRY(cudaSetDevice(ordinal));
    const int variant = gemm_variant_for(m);
    CUtensorMap ma, mb, mc;
    rc = make_map(&ma, a, m, k, variant == 3 ? 2 * BM : BM);
    if (rc) return rc;
    rc = make_map(&mb, b, n, k, variant == 1 ? BN : BN / 2);
    if (rc) return rc;
    rc = make_map(&mc, c, m, n, 32, variant == 3 ? 32 : EPI_UNIT_COLS);      // one tensor store = 32 rows x 64 (variant 3: 32) columns
    if (rc) return rc;
    if (variant == 3) {
        B200_CUDA_TRY(cudaFuncSetAttribute(gemm_bf16_tn_2cta_512_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM3_BYTES));
        const int tiles = ((m + 4 * BM - 1) / (4 * BM)) * (n / BN);
        const int pairs = std::min(tiles, props.sms / 2);
        GemmTune tune = kShippedTune3;          // bands of 4 x 512 rows (the same 2048 rows as the 256 x 256 kernel's bands)
        if (const char* e = getenv("B200PROBE_GEMM_PREFETCH")) { int v = atoi(e); if (v >= 0 && v <= 64) tune.prefetch = v; }
        if (const char* e = getenv("B200PROBE_GEMM_EXPT")) tune.expt = atoi(e);
        if (const char* e = getenv("B200PROBE_GEMM_EPI")) tune.epi = atoi(e);
        if (const char* e = getenv("B200PROBE_GEMM_SKEW")) tune.skew = atoi(e);
        if (const char* e = getenv("B200PROBE_GEMM_GROUP_M")) { int v = atoi(e); if (v >= 1 && v <= 64) tune.group_m = v; }
        if (const char* e = getenv("B200PROBE_GEMM_POL_A")) tune.pol_a = atoi(e);
        if (const char* e = getenv("B200PROBE_GEMM_POL_B")) tune.pol_b = atoi(e);
        if (const char* e = getenv("B200PROBE_GEMM_POL_C")) tune.pol_c = atoi(e);
        gemm_bf16_tn_2cta_512_kernel<<<2 * pairs, NUM_THREADS3, SMEM3_BYTES, (cudaStream_t)stream>>>(ma, mb, mc, (__nv_bfloat16*)c, m, n, k, tune);
    } else if (variant == 2) {
        B200_CUDA_TRY(cudaFuncSetAttribute(gemm_bf16_tn_2cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM2_BYTES));
        const int tiles = (m / (2 * BM)) * (n / BN);
        const int pairs = std::min(tiles, props.sms / 2);
        GemmTune tune{GROUP_M / 2, 0, 0, 0, 0, 0, 0, 0};
        if (const char* e = getenv("B200PROBE_GEMM_GROUP_M")) { int v = atoi(e); if (v >= 1 && v <= 64) tune.group_m = v; }
        if (const char* e = getenv("B200PROBE_GEMM_POL_A")) tune.pol_a = atoi(e);
        if (const char* e = getenv("B200PROBE_GEMM_POL_B")) tune.pol_b = atoi(e);
        if (const char* e = getenv("B200PROBE_GEMM_POL_C")) tune.pol_c = atoi(e);
        gemm_bf16_tn_2cta_kernel<<<2 * pairs, NUM_THREADS, SMEM2_BYTES, (cudaStream_t)stream>>>(ma, mb, mc, m, n, k, tune);
    } else {
        B200_CUDA_TRY(cudaFuncSetAttribute(gemm_bf16_tn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        const int tiles = (m / BM) * (n / BN);
        const int grid = std::min(tiles, props.sms);
        gemm_bf16_tn_kernel<<<grid, NUM_THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(ma, mb, mc, m, n, k);
    }
    B200_CUDA_TRY(cudaGetLastError());
    return 0;
}

int b200probe_gemm_fp8_launch(int ordinal, const void* a, const void* b, void* c, int m, int n, int k, void* stream) {
    b200::DevProps props;
    int rc = b200::device_props(ordinal, &props);
    if (rc) return rc;
    rc = check_shape_fp8(m, n, k);
    if (rc) return rc;
    if (!a || !b || !c || (((uintptr_t)a | (uintptr_t)b | (uintptr_t)c) & 15)) { b200::set_error("gemm_fp8: operands must be 16-byte aligned device pointers"); return B200PROBE_EINVAL; }
    B200_CUDA_TRY(cudaSetDevice(ordinal));
    CUtensorMap ma, mb;
    rc = make_map(&ma, a, m, k, 2 * BM, OperandE4m3::kKbElems, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1);
    if (rc) return rc;
    rc = make_map(&mb, b, n, k, BN / 2, OperandE4m3::kKbElems, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1);
    if (rc) return rc;
    B200_CUDA_TRY(cudaFuncSetAttribute(gemm_e4m3_tn_2cta_512_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM3_BYTES));
    const int tiles = ((m + 4 * BM - 1) / (4 * BM)) * (n / BN);
    const int pairs = std::min(tiles, props.sms / 2);
    gemm_e4m3_tn_2cta_512_kernel<<<2 * pairs, NUM_THREADS3, SMEM3_BYTES, (cudaStream_t)stream>>>(ma, mb, (__nv_bfloat16*)c, m, n, k);
    B200_CUDA_TRY(cudaGetLastError());
    return 0;
}

int b200probe_gemm_release(int ordinal) {
    if (ordinal < 0 || ordinal >= B200PROBE_MAX_DEVICES) return B200PROBE_ERANGE;
    GemmArena& g = g_gemm[ordinal];
    GemmLock lock(g);
    if (g.stream) { cudaSetDevice(ordinal); gemm_arena_free(g); }
    return 0;
}

// e4m3 = 0: the bf16 kernels (b200probe_gemm), 1: the E4M3 kernel (b200probe_gemm_fp8); the same protocol and verdict rules
static int gemm_locked(int ordinal, GemmArena& g, const b200probe_gemm_cfg_t& cfg, int e4m3, b200probe_gemm_result_t* out) {
    const int M = cfg.m, N = cfg.n, K = cfg.k, S = cfg.samples;
    const int cls = cfg.operands;
    const int kind = (e4m3 ? 4 : 0) | (cls << 1);                   // b200probe_gemm_fill's `which` without the matrix bit
    auto launch = [&]() { return e4m3 ? b200probe_gemm_fp8_launch(ordinal, g.a, g.b, g.c, M, N, K, g.stream) : b200probe_gemm_launch(ordinal, g.a, g.b, g.c, M, N, K, g.stream); };
    auto value = [&](uint64_t e, int mat) {
        const uint16_t v = b200probe_gemm_operand_bits(e, cfg.seed, kind | mat);
        return e4m3 ? e4m3_bits_to_double((uint8_t)v) : (double)bf16_bits_to_float(v);
    };
    int rc = gemm_arena_reserve(g, M, N, K, S);
    if (rc) return rc;
    if (!g.filled || g.seed != cfg.seed || g.operands != cls || g.e4m3 != e4m3) {
        rc = b200probe_gemm_fill(ordinal, g.a, (uint64_t)M * K, cfg.seed, kind | 0, g.stream);
        if (rc) return rc;
        rc = b200probe_gemm_fill(ordinal, g.b, (uint64_t)N * K, cfg.seed, kind | 1, g.stream);
        if (rc) return rc;
        g.filled = true; g.seed = cfg.seed; g.operands = cls; g.e4m3 = e4m3;
    }
    B200_CUDA_TRY(cudaMemsetAsync(g.c, 0xFF, (size_t)M * N * 2, g.stream));      // poison: a tile the kernel skipped cannot pass the check

    std::vector<float> ms((size_t)cfg.reps);
    for (int it = -cfg.warmup; it < cfg.reps; ++it) {
        if (it >= 0) B200_CUDA_TRY(cudaEventRecord(g.e0, g.stream));
        rc = launch();
        if (rc) return rc;
        if (it >= 0) {
            B200_CUDA_TRY(cudaEventRecord(g.e1, g.stream));
            B200_CUDA_TRY(cudaEventSynchronize(g.e1));
            B200_CUDA_TRY(cudaEventElapsedTime(&ms[it], g.e0, g.e1));
        }
    }
    B200_CUDA_TRY(cudaStreamSynchronize(g.stream));
    const double flop = 2.0 * M * N * (double)K;
    out->ms_median = median_f(ms);
    out->ms_best = *std::min_element(ms.begin(), ms.end());
    out->tflops_median = flop / (out->ms_median * 1e-3) / 1e12;
    out->tflops_best = flop / (out->ms_best * 1e-3) / 1e12;

    if (cfg.sustain_seconds > 0) {
        // back-to-back launches for the requested wall time (power-capped steady state)
        int batch = std::max(1, (int)(0.25 / (out->ms_median * 1e-3)));
        double total_ms = 0, total_n = 0;
        while (total_ms * 1e-3 < cfg.sustain_seconds) {
            float t;
            B200_CUDA_TRY(cudaEventRecord(g.e0, g.stream));
            for (int i = 0; i < batch; ++i) {
                rc = launch();
                if (rc) return rc;
            }
            B200_CUDA_TRY(cudaEventRecord(g.e1, g.stream));
            B200_CUDA_TRY(cudaEventSynchronize(g.e1));
            B200_CUDA_TRY(cudaEventElapsedTime(&t, g.e0, g.e1));
            total_ms += t; total_n += batch;
        }
        out->tflops_sustained = flop * total_n / (total_ms * 1e-3) / 1e12;
    }

    // data result: checksum of C (run-to-run identity) + sampled outputs against fp64 dot products
    B200_CUDA_TRY(cudaMemsetAsync(g.partials, 0, 16, g.stream));
    rc = b200probe_hbm_read(ordinal, g.c, (uint64_t)M * N * 2, (uint64_t*)g.partials, nullptr, g.stream);
    if (rc) return rc;
    unsigned long long h[2];
    B200_CUDA_TRY(cudaMemcpyAsync(h, g.partials, 16, cudaMemcpyDeviceToHost, g.stream));
    std::vector<uint64_t> idxs((size_t)S);
    for (int i = 0; i < S; ++i) {
        // corners and tile seams first, then a hash-scattered set
        uint32_t r, c;
        if (i < 4) { r = (i & 1) ? M - 1 : 0; c = (i & 2) ? N - 1 : 0; }
        else if (i < 8) { r = (i & 1) ? BM : BM - 1; c = (i & 2) ? BN : BN - 1; r = std::min<uint32_t>(r, M - 1); c = std::min<uint32_t>(c, N - 1); }
        else { r = b200_mix32(cfg.seed ^ (0x9E37u * i)) % (uint32_t)M; c = b200_mix32(cfg.seed + 77u * i + 1) % (uint32_t)N; }
        idxs[i] = (uint64_t)r * N + c;
    }
    B200_CUDA_TRY(cudaMemcpyAsync(g.idx, idxs.data(), (size_t)S * 8, cudaMemcpyHostToDevice, g.stream));
    gather_kernel<<<(S + 255) / 256, 256, 0, g.stream>>>((const uint16_t*)g.c, (const uint64_t*)g.idx, (uint16_t*)g.out, S);
    B200_CUDA_TRY(cudaGetLastError());
    std::vector<uint16_t> got((size_t)S);
    B200_CUDA_TRY(cudaMemcpyAsync(got.data(), g.out, (size_t)S * 2, cudaMemcpyDeviceToHost, g.stream));
    B200_CUDA_TRY(cudaStreamSynchronize(g.stream));
    out->c_sum64 = h[0];
    out->c_xor32 = (uint32_t)h[1];
    int bad = 0;
    double max_abs = 0, max_rel = 0, max_over_tol = 0;
    const double acc_allow = ldexp(sqrt((double)K), -10);      // UNIFORM: fp32 accumulation allowance, 2^-10 sqrt(K)
    for (int i = 0; i < S; ++i) {
        const uint64_t r = idxs[i] / N, c = idxs[i] % N;
        double acc = 0;
        for (int k = 0; k < K; ++k)
            acc += value(r * K + k, 0) * value(c * K + k, 1);
        const double gotf = bf16_bits_to_float(got[i]);
        const double err = fabs(gotf - acc);
        max_abs = std::max(max_abs, err);
        if (acc != 0) max_rel = std::max(max_rel, err / fabs(acc));
        if (cls == B200PROBE_GEMM_OPERANDS_EXACT) {
            if (got[i] != float_to_bf16_rne((float)acc)) ++bad;      // bit-exact bar: operands make every partial sum exact in fp32
        } else {
            const double tol = ldexp(fabs(acc), -8) + acc_allow;      // half a bf16 ulp of the result + the accumulation allowance
            max_over_tol = std::max(max_over_tol, err / tol);
            if (!(err <= tol)) ++bad;                                 // also catches NaN
        }
    }
    out->samples = S; out->bad = bad;
    out->max_abs_err = max_abs; out->max_rel_err = max_rel; out->max_err_over_tol = max_over_tol;
    out->verified = bad == 0 ? 1 : 0;
    if (bad) {
        b200::set_error("%s: %d of %d sampled outputs %s (max abs err %g)", e4m3 ? "gemm_fp8" : "gemm", bad, S,
                        cls == B200PROBE_GEMM_OPERANDS_EXACT ? "differ from the fp64 contraction rounded to bf16" : "are outside 2^-8|ref| + 2^-10 sqrt(K) of the fp64 contraction", max_abs);
        return B200PROBE_EMISMATCH;
    }
    return 0;
}

static int gemm_entry(int idx, const b200probe_gemm_cfg_t* cfg_in, int e4m3, b200probe_gemm_result_t* out) {
    if (!out) return B200PROBE_EINVAL;
    int ordinal = -1;
    int rc = b200::cuda_ordinal_of(idx, &ordinal);
    if (rc) return rc;
    b200::DevProps props;
    rc = b200::device_props(ordinal, &props);
    if (rc) return rc;
    b200probe_gemm_cfg_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    if (cfg_in) cfg = *cfg_in;
    if (!cfg.m) cfg.m = 8192;
    if (!cfg.n) cfg.n = 8192;
    if (!cfg.k) cfg.k = 8192;
    if (!cfg.warmup && !cfg.reps) { cfg.warmup = 3; cfg.reps = 10; }
    if (cfg.reps < 1) cfg.reps = 1;
    if (!cfg.seed) cfg.seed = 0xB200u;
    if (!cfg.samples) cfg.samples = 1024;
    if (cfg.samples < 1 || cfg.samples > (1 << 20)) { b200::set_error("gemm: samples out of range"); return B200PROBE_EINVAL; }
    if (cfg.operands != B200PROBE_GEMM_OPERANDS_EXACT && cfg.operands != B200PROBE_GEMM_OPERANDS_UNIFORM) { b200::set_error("gemm: unknown operand class %d", cfg.operands); return B200PROBE_EINVAL; }
    rc = e4m3 ? check_shape_fp8(cfg.m, cfg.n, cfg.k) : check_shape(cfg.m, cfg.n, cfg.k);
    if (rc) return rc;
    memset(out, 0, sizeof(*out));
    out->m = cfg.m; out->n = cfg.n; out->k = cfg.k;
    out->operands = cfg.operands;
    out->verified = -1;
    B200_CUDA_TRY(cudaSetDevice(ordinal));
    GemmArena& g = g_gemm[ordinal];
    GemmLock lock(g);
    rc = gemm_locked(ordinal, g, cfg, e4m3, out);
    if (rc && rc != B200PROBE_EMISMATCH) gemm_arena_free(g);      // unknown state after a CUDA error / failed allocation: start over next time
    return rc;
}

int b200probe_gemm(int idx, const b200probe_gemm_cfg_t* cfg_in, b200probe_gemm_result_t* out) { return gemm_entry(idx, cfg_in, 0, out); }

int b200probe_gemm_fp8(int idx, const b200probe_gemm_cfg_t* cfg_in, b200probe_gemm_result_t* out) { return gemm_entry(idx, cfg_in, 1, out); }

}  // extern "C"
