/*
 * b200probe.h — C ABI of libb200probe.so, the B200-native active health-probe engine.
 *
 * This is the drop-in boundary (SURVEY.md §8b "Inner"): the exact surface a device-plugin host
 * (Go via cgo, Python via ctypes, the bench harness, the tests) binds.  extern "C", plain pointers
 * and sizes, caller-allocated out-buffers, no callbacks, no C++ or torch types.
 *
 * What each group replaces in the reference stack (the reference repo holds no code; it installs
 * the un-pinned NVIDIA k8s-device-plugin chart — /root/reference/README.md:109,116 — configured by
 * /root/reference/values.yaml:1-18; upstream internals are cited from recall and marked [RECALLED]):
 *
 *   b200probe_device_*      -> the plugin's NVML enumeration that backs ListAndWatch
 *                              (values.yaml:16-18 selects the resource; nvml.h:4063,4131,4616,4274,6110,6161)
 *   b200probe_health_*      -> the plugin's passive XID/ECC event loop [RECALLED checkHealth];
 *                              NVML entry points nvml.h:9125 (EventSetCreate), :9161 (RegisterEvents),
 *                              :9222 (EventSetWait_v2).  north_star calls this "nvmlDeviceGetHealth";
 *                              no such NVML call exists (SURVEY.md §0 fact 3).
 *   b200probe_hbm_*         -> NEW: no reference counterpart (SURVEY.md §8a row a11)
 *   b200probe_a2a_*         -> NEW: row a12
 *   b200probe_gemm*         -> NEW: row a13
 *   b200probe_gemm_fp8*     -> NEW: row a15 (FP8 tensor cores, DESIGN.md §4.5)
 *   b200probe_hbm_memtest,
 *   b200probe_memtest_element,
 *   b200probe_hbm_ecc       -> NEW: HBM integrity (DESIGN.md §4.4)
 *
 * Error convention: 0 = OK; negative = library error (B200PROBE_E*); positive = a foreign status
 * tagged by range: 1000+cudaError_t, 2000+nvmlReturn_t, 3000+ncclResult_t.
 * b200probe_strerror() never returns NULL.  b200probe_last_error() returns the calling thread's
 * most recent detailed message.
 *
 * Threading: every call is re-entrant per device index; each probe call sets its own device and
 * uses its own stream unless one is passed.  The a2a calls are the only cross-device calls and
 * serialise internally.  A Go caller must runtime.LockOSThread() around a call (CUDA's current
 * device is per OS thread).
 */
#ifndef B200PROBE_H_
#define B200PROBE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200PROBE_ABI_VERSION 2

/* ---- status codes --------------------------------------------------------------------------- */
#define B200PROBE_OK            0
#define B200PROBE_EINVAL       (-1)   /* bad argument                                             */
#define B200PROBE_ENOTINIT     (-2)   /* b200probe_init not called                                */
#define B200PROBE_ENVML        (-3)   /* libnvidia-ml could not be loaded / symbol missing        */
#define B200PROBE_ENOCUDA      (-4)   /* no CUDA device / driver; the probes never fall back to CPU */
#define B200PROBE_ERANGE       (-5)   /* out-buffer too small / index out of range                */
#define B200PROBE_EMISMATCH    (-6)   /* data verification failed (checksum / numeric check)      */
#define B200PROBE_ENOPEER      (-7)   /* peer access between the requested devices is unavailable */
#define B200PROBE_ENONCCL      (-8)   /* libnccl could not be loaded                              */
#define B200PROBE_EARCH        (-9)   /* device is not sm_100 (kernels are sm_100a-only)          */
#define B200PROBE_ENOMEM       (-10)
#define B200PROBE_ESTATE       (-11)  /* call sequence error (e.g. health poll before open)       */
#define B200PROBE_CUDA_BASE    1000
#define B200PROBE_NVML_BASE    2000
#define B200PROBE_NCCL_BASE    3000

#define B200PROBE_MAX_DEVICES  64

/* ---- lifecycle ------------------------------------------------------------------------------ */
int         b200probe_abi_version(void);
/* dlopen NVML (nvml_path_or_null, else $B200PROBE_NVML_PATH, else "libnvidia-ml.so.1") and
 * nvmlInit_v2.  CUDA is initialised lazily by the first probe call, so enumeration and passive
 * health work in a process that never touches CUDA (exactly like the reference plugin). */
int         b200probe_init(const char* nvml_path_or_null);
void        b200probe_shutdown(void);
const char* b200probe_strerror(int rc);
int         b200probe_last_error(char* buf, int cap);

/* ---- enumeration (NVML order == the order the reference plugin advertises) -------------------- */
typedef struct b200probe_device {
    int      index;                 /* NVML index                                                  */
    char     uuid[96];              /* "GPU-xxxxxxxx-…"  (NVML_DEVICE_UUID_V2_BUFFER_SIZE)         */
    char     name[96];
    char     pci_bus_id[32];
    uint64_t mem_total;             /* bytes, nvmlDeviceGetMemoryInfo().total                      */
    int      cc_major, cc_minor;
    int      numa_node;             /* -1 when NVML reports NOT_SUPPORTED                          */
    int      mig_enabled;           /* current MIG mode; -1 when not supported                     */
    uint64_t supported_events;      /* nvmlDeviceGetSupportedEventTypes                            */
    int      cuda_ordinal;          /* CUDA ordinal with the same UUID, -1 if CUDA not initialised
                                       or the device is hidden by CUDA_VISIBLE_DEVICES             */
} b200probe_device_t;

int b200probe_device_count(int* n);
int b200probe_device_info(int idx, b200probe_device_t* out);
/* Microseconds the last full enumerate took (timed inside the library, CLOCK_MONOTONIC). */
int b200probe_enumerate(b200probe_device_t* out, int cap, int* n, double* usec);

/* ---- passive health: twin of the reference plugin's XID/ECC event loop ------------------------ */
typedef struct b200probe_health_event {
    int      rc_wait;               /* raw nvmlReturn_t of the wait (0 success, 10 timeout …)      */
    uint64_t event_type;            /* nvmlEventData_t.eventType                                   */
    uint64_t event_data;            /* XID number for XidCriticalError                             */
    uint32_t gpu_instance_id, compute_instance_id;
    int      device_index;          /* -1 when the UUID of the event's device is unreadable        */
    int      skipped;               /* 1 = non-XID event or XID on the skip list (stays healthy)   */
    uint64_t newly_unhealthy;       /* bit i = device i turned Unhealthy because of this event     */
} b200probe_health_event_t;

/* disable_healthchecks mirrors env DP_DISABLE_HEALTHCHECKS [RECALLED]: NULL/"" = default skip
 * list {13,31,43,45,68,109}; "all" or containing "xids" = loop disabled (every device stays
 * Healthy); otherwise a comma list of extra XIDs to skip.  unhealthy_at_open gets the devices
 * that could not be registered (marked Unhealthy at registration, like the reference). */
int  b200probe_health_open(const char* disable_healthchecks, uint64_t* unhealthy_at_open);
/* One nvmlEventSetWait_v2(timeout_ms).  Returns OK on timeout too (ev->rc_wait == 10). */
int  b200probe_health_wait(int timeout_ms, b200probe_health_event_t* ev);
/* Survey-proposed one-shot form: open if needed, wait once, return the sticky unhealthy mask
 * (there is no path back to Healthy, as in the reference). */
int  b200probe_passive_health(int timeout_ms, uint64_t* unhealthy_mask);
int  b200probe_health_mask(uint64_t* unhealthy_mask);
void b200probe_health_close(void);

/* ---- is the device in use by somebody else? ------------------------------------------------------
 * The active probes are gated against idle-box figures and compete with tenants for SMs, HBM bandwidth and
 * memory (values.yaml:16-18 time-slices every GPU four ways, so tenants are the normal case).  The host asks
 * before a probe round and SKIPS a busy device (verdict "inconclusive", last idle verdict kept) — it never
 * reports a loaded GPU as unhealthy.  compute_procs excludes the calling process (NVML reports host-namespace
 * pids: a caller that has probed the device and cannot find its own pid is assumed to be one of the entries). */
#define B200PROBE_BUSY_UTIL_PCT 10
typedef struct b200probe_busy {
    int      compute_procs;         /* nvmlDeviceGetComputeRunningProcesses_v3 minus this process; -1 = unreadable */
    int      util_gpu_pct, util_mem_pct;   /* nvmlDeviceGetUtilizationRates (last sample period); -1 = unreadable  */
    uint64_t mem_used;              /* nvmlDeviceGetMemoryInfo().used, bytes                                         */
    int      busy;                  /* compute_procs > 0 || util_gpu_pct >= B200PROBE_BUSY_UTIL_PCT                  */
} b200probe_busy_t;
int b200probe_device_busy(int idx, b200probe_busy_t* out);

/* ---- passive NVLink / fabric status (SURVEY.md §8f.3) ------------------------------------------- */
typedef struct b200probe_nvlink_status {
    int      links_total;           /* links NVML reports a state for (18 on a B200)               */
    int      links_active;
    uint32_t active_mask;           /* bit l = link l is up                                        */
    int      fabric_state;          /* nvmlGpuFabricState_t (3 = completed); -1 = not supported    */
    int      fabric_status;         /* nvmlReturn_t of the fabric registration                     */
    uint32_t fabric_health_mask;
    uint64_t data_tx_kib, data_rx_kib;   /* payload counters, summed over links, since driver load */
    uint64_t raw_tx_kib, raw_rx_kib;     /* payload + protocol overhead                            */
    int      counters_ok;
} b200probe_nvlink_status_t;
int b200probe_nvlink_passive(int idx, b200probe_nvlink_status_t* out);

/* ---- HBM bandwidth sweep (row a11) ------------------------------------------------------------ */
#define B200PROBE_HBM_READ   1
#define B200PROBE_HBM_WRITE  2
#define B200PROBE_HBM_COPY   4
/* kernel variants */
#define B200PROBE_VARIANT_TMA     0   /* cp.async.bulk global<->shared ring + mbarrier (default)   */
#define B200PROBE_VARIANT_DIRECT  1   /* LDG.128/STG.128 grid-stride                               */

typedef struct b200probe_hbm_cfg {
    uint64_t min_bytes, max_bytes;  /* powers of two inclusive; 0,0 = 1 MiB … 1 GiB               */
    int      modes;                 /* bitmask of B200PROBE_HBM_*; 0 = all three                   */
    int      warmup, reps;          /* 0,0 = 3,20                                                  */
    uint32_t seed;                  /* 0 = 0xB200                                                  */
    int      variant;
    int      verify;                /* 1 = check every data result against the closed-form pattern */
    int      flush_l2;              /* 1 = overwrite a >L2 scratch between timed reps              */
    /* tuning (0 = built-in default) */
    int      stage_bytes, stages, warps_per_cta, ctas_per_sm;
    int      launches_per_rep;      /* launches between the two events of one timed rep: 0 = about a
                                       millisecond of work (the kernel's rate, not launch latency),
                                       1 = single launches                                          */
} b200probe_hbm_cfg_t;

typedef struct b200probe_hbm_result {
    uint64_t bytes;                 /* buffer size N                                               */
    int      mode, variant;
    double   ms_median, ms_best;
    double   gbs_median, gbs_best;  /* algorithmic bytes (N read, N write, 2N copy) / time, 1e9 B/s */
    uint64_t sum64;                 /* data result: sum of u32 words mod 2^64 …                    */
    uint32_t xor32;                 /* … and xor of u32 words, of the buffer the mode produced/read */
    int      verified;              /* 1 = every word equals the regenerated pattern (device-side
                                       compare), 0 = mismatch, -1 not checked                      */
    int      cache_resident;        /* 1 = footprint fits L2: reported, never used for the verdict */
} b200probe_hbm_result_t;

int b200probe_hbm_sweep(int idx, const b200probe_hbm_cfg_t* cfg,
                        b200probe_hbm_result_t* out, int cap, int* n);
/* The sweep keeps its two device buffers, stream and events resident per device between calls
 * (the plugin probes periodically).  Release them explicitly; b200probe_shutdown does not touch
 * CUDA state. */
int b200probe_hbm_release(int cuda_ordinal);

/* Resident-buffer launchers (bench / tests / plugin reuse).  Pointers are DEVICE pointers of
 * device cuda_ordinal; stream is a cudaStream_t (NULL = legacy default stream).  bytes must be a
 * multiple of 4; pointers 16-byte aligned.  Asynchronous: returns after the launch.
 *   fill : dst[i] = pattern(i, seed)                      (write mode)
 *   copy : dst[i] = src[i]                                (copy mode)
 *   read : partials[0..1] += (sum64, xor32) of src        (read mode; partials = 2 x u64 on device,
 *          zeroed by the caller; reduction is commutative so the result is launch-order exact)  */
int b200probe_hbm_fill (int cuda_ordinal, void* dst, uint64_t bytes, uint32_t seed,
                        const b200probe_hbm_cfg_t* tuning_or_null, void* stream);
int b200probe_hbm_copy (int cuda_ordinal, const void* src, void* dst, uint64_t bytes,
                        const b200probe_hbm_cfg_t* tuning_or_null, void* stream);
int b200probe_hbm_read (int cuda_ordinal, const void* src, uint64_t bytes, uint64_t* partials,
                        const b200probe_hbm_cfg_t* tuning_or_null, void* stream);
/* The probe's verdict pass on any device buffer: checksum (sum64, xor32 of the u32 words) plus a
 * device-side compare with the closed-form pattern under `seed`: number of words that differ and the
 * index of the lowest one (~0 when none).  TMA-staged like the read sweep.  Synchronous. */
int b200probe_hbm_verify(int cuda_ordinal, const void* buf, uint64_t bytes, uint32_t seed,
                         uint64_t* sum64, uint32_t* xor32, uint64_t* bad_words, uint64_t* first_bad_word);
/* Host-buffer entry (the data-carrying e2e form): src_host -> H2D -> copy kernel -> checksum of what
 * landed -> D2H into dst_host, pipelined over 8 MiB chunks on three streams so both PCIe directions
 * and the kernel overlap.  Any host memory works; pinned buffers from b200probe_host_alloc reach the
 * PCIe rate (pageable ones are staged by the driver).  Synchronous. */
int b200probe_hbm_copy_host(int cuda_ordinal, const void* src_host, void* dst_host, uint64_t bytes,
                            uint64_t* sum64, uint32_t* xor32);
/* Page-locked host memory for the entry above (cudaHostAlloc, portable across devices). */
int b200probe_host_alloc(uint64_t bytes, void** ptr);
int b200probe_host_free(void* ptr);

/* ---- HBM integrity: march test over the free memory, joined with NVML ECC / row-remap state ------- */
/* Passive side.  Every field is -1 when NVML does not support or does not export the query. */
typedef struct b200probe_ecc_status {
    int      ecc_mode;              /* nvmlDeviceGetEccMode, current: 1 enabled, 0 disabled          */
    int64_t  corrected_volatile;    /* nvmlDeviceGetTotalEccErrors(CORRECTED, VOLATILE): since driver load */
    int64_t  uncorrected_volatile;  /* nvmlDeviceGetTotalEccErrors(UNCORRECTED, VOLATILE)           */
    int      remap_corrected_rows;  /* nvmlDeviceGetRemappedRows: rows remapped for corrected errors */
    int      remap_uncorrected_rows;/* … for uncorrected errors                                     */
    int      remap_pending;         /* 1 = a remap waits for the next GPU reset                      */
    int      remap_failure;         /* 1 = a remap failed (no spare row left)                        */
} b200probe_ecc_status_t;
int b200probe_hbm_ecc(int idx, b200probe_ecc_status_t* out);

/* One march element over a device buffer of device cuda_ordinal, for every u32 word i:
 *   VERIFY: compare buf[i] with pattern(base_word + i, expect_seed);
 *   WRITE : then store pattern(base_word + i, write_seed) in place.
 * base_word places the buffer in a larger tested space (address-in-address across chunks); the
 * complement of a pattern is the pattern under seed ^ 0xFFFFFFFF.  bytes a multiple of 4, buf
 * 16-byte aligned.  Mismatches: count, lowest global word index (~0 when none) and the OR of
 * got ^ want over all of them.  Synchronous; holds no device memory after it returns. */
#define B200PROBE_MEMTEST_VERIFY 1
#define B200PROBE_MEMTEST_WRITE  2
int b200probe_memtest_element(int cuda_ordinal, void* buf, uint64_t bytes, uint64_t base_word, int flags,
                              uint32_t expect_seed, uint32_t write_seed,
                              uint64_t* bad_words, uint64_t* first_bad_word, uint32_t* bad_bits);

typedef struct b200probe_memtest_cfg {
    double   fraction;              /* of cudaMemGetInfo's free bytes, in (0, 1]; 0 = 0.9          */
    uint64_t max_bytes;             /* cap on the bytes tested; 0 = none                           */
    uint64_t min_bytes;             /* fewer bytes allocated -> B200PROBE_ENOMEM; 0 = one byte      */
    uint64_t chunk_bytes;           /* allocation unit, multiple of 4096; 0 = 1 GiB                 */
    int      passes;                /* 0 = 1                                                       */
    uint32_t seed;                  /* s0; 0 = 0xB200.  s1 = s0 ^ 0x5A5A5A5A                       */
} b200probe_memtest_cfg_t;

typedef struct b200probe_memtest_result {
    uint64_t bytes_tested;
    int      chunks, passes;
    uint64_t free_before, total;    /* cudaMemGetInfo before the allocation                         */
    double   alloc_ms, test_ms;     /* allocation (host clock); all elements of all passes (events) */
    double   gbs;                   /* algorithmic bytes (6 x bytes_tested per pass) / test_ms      */
    uint64_t bad_words;             /* mismatching words, summed over the verifying elements        */
    uint64_t first_bad_word;        /* lowest mismatching word index (in the tested space) of the
                                       first element that saw one; ~0 when none                    */
    uint32_t bad_bits;              /* OR of got ^ want over every mismatch                          */
    int      first_bad_element;     /* 1, 2 or 3 (E1..E3) of that element; -1 when none            */
    int64_t  ecc_corrected_delta;   /* volatile ECC totals after - before; -1 when unreadable       */
    int64_t  ecc_uncorrected_delta;
    b200probe_ecc_status_t ecc_after;
} b200probe_memtest_result_t;

/* The HBM integrity probe on NVML device idx: ECC snapshot; allocate fraction x free (capped by
 * max_bytes) in chunk_bytes pieces, stopping at the first failed allocation; march
 *   E0 write P(s0); E1 verify P(s0), write ~P(s0); E2 verify ~P(s0), write P(s1); E3 verify P(s1)
 * with every element over all chunks before the next one, `passes` times; ECC snapshot; free.
 * Nothing stays allocated after the call, on any path.  Less than min_bytes allocated returns
 * B200PROBE_ENOMEM (a resource verdict, not a fault); mismatches are results, not errors. */
int b200probe_hbm_memtest(int idx, const b200probe_memtest_cfg_t* cfg, b200probe_memtest_result_t* out);

/* ---- NVLink all-to-all (row a12) --------------------------------------------------------------- */
#define B200PROBE_A2A_PEER_ALL    0   /* our peer-memory kernel, all pairs concurrently            */
#define B200PROBE_A2A_PEER_PAIR   1   /* same kernel, one (src,dst) pair at a time -> matrix       */
#define B200PROBE_A2A_NCCL        2   /* grouped ncclSend/ncclRecv (the library leg, for contrast) */
#define B200PROBE_A2A_CE          3   /* cudaMemcpyPeerAsync of every chunk (copy engines; the second
                                         library leg: the two-way peer-copy rate measured in the same run) */
/* exchange kernels (cfg.variant) */
#define B200PROBE_A2A_AUTO        0   /* one pair: PULL_TMA; concurrent exchange: PUSH_SYNC when G > 2 and
                                         S >= 64 MiB (128 MiB for free-running launches), else PUSH_TMA */
#define B200PROBE_A2A_PULL_TMA    1   /* bulk-LOAD the peers' send chunks over NVLink: best one-way
                                         (756-781 GB/s), worse when both directions are loaded (626) */
#define B200PROBE_A2A_PUSH_TMA    2   /* generate in shared memory, bulk-STORE into the peers: best
                                         for the all-to-all (692 GB/s per direction per GPU)         */
#define B200PROBE_A2A_PUSH_DIRECT 3   /* generate in registers, 16-byte stores on peer pointers     */
#define B200PROBE_A2A_PUSH_BUF    4   /* bulk-load the local send chunk, bulk-store into the peer   */
#define B200PROBE_A2A_MIX_TMA     5   /* each chunk moved from both ends: head pushed by its source,
                                         tail pulled by its destination ($B200PROBE_A2A_MIX_PCT)     */

#define B200PROBE_A2A_PUSH_STAGGER 6  /* PUSH_TMA with the peers visited one at a time, rank r sending to
                                         (r+t) mod G at step t: one source per destination at a time */

#define B200PROBE_A2A_PUSH_SYNC    7  /* PUSH_STAGGER + a device-side barrier over all ranks before every
                                         step (relaxed flags in the windows' sync pages, written over
                                         NVLink): 701 GB/s per direction at G = 8 vs 618-660 free-running */

typedef struct b200probe_a2a_cfg {
    uint64_t bytes_per_pair;        /* S, multiple of 16; 0 = 256 MiB                              */
    int      mode;
    int      warmup, reps;          /* 0,0 = 2,10                                                  */
    uint32_t seed;
    int      verify;
    int      ctas_per_peer;         /* 0 = default (about one CTA per SM in total)                 */
    int      variant;               /* B200PROBE_A2A_AUTO ...                                      */
} b200probe_a2a_cfg_t;

typedef struct b200probe_a2a_result {
    int      g;
    double   ms_median, ms_best;    /* of the all-pairs exchange (modes 0, 2), max over devices     */
    double   egress_gbs[B200PROBE_MAX_DEVICES];   /* (G-1)*S / t per GPU, payload bytes            */
    double   ingress_gbs[B200PROBE_MAX_DEVICES];
    double   min_pair_gbs, max_pair_gbs;
    int      verified;              /* 1 = every landed chunk equals the regenerated pattern        */
    int      pair_source;           /* what pair_gbs holds: B200PROBE_PAIR_*                        */
} b200probe_a2a_result_t;
#define B200PROBE_PAIR_SHARE     0    /* egress / (g-1): the pair's share of a concurrent exchange    */
#define B200PROBE_PAIR_ISOLATED  1    /* PEER_PAIR: the pair moved alone on an otherwise idle fabric  */
#define B200PROBE_PAIR_STEPPED   2    /* PUSH_SYNC steps, each DRAINED before the next: S / (last store
                                         complete - step start), every rank busy with one pair       */

/* Single process, all GPUs (how the plugin daemon runs).  cuda_ordinals[g]; pair_gbs is g*g
 * row-major [src][dst], diagonal 0.  PEER_PAIR: each pair measured alone.  PEER_ALL: under PUSH_SYNC
 * the exchange moves one pair per step (src -> (src+t) mod g); after the timed exchanges three more
 * run with every step drained and time-stamped on the device, and the entry is the median of that
 * pair's own rate, first byte issued to last store complete (never above the port rate); for the
 * free-running schedules it is the pair's share egress/(g-1).  out->pair_source says which.
 * Windows, streams and NCCL communicators stay resident between calls with the same devices, S and
 * seed; b200probe_a2a_release() frees them (the plugin does after every probe round).
 * A failed device allocation returns B200PROBE_ENOMEM (a resource verdict, not a fault). */
int b200probe_nvlink_a2a(const int* cuda_ordinals, int g, const b200probe_a2a_cfg_t* cfg,
                         double* pair_gbs, b200probe_a2a_result_t* out);
int b200probe_a2a_release(void);

/* Enable peer access between every ordered pair of the listed devices (idempotent). */
int b200probe_enable_peer_access(const int* cuda_ordinals, int g);

/* Building blocks (one process per GPU under torchrun, or a host that owns its windows).
 * Window layout on every rank:  [recv: world x S][send: world x S][sync page]  bytes;
 *   send[p] = this rank's chunk for rank p, recv[p] = where rank p's chunk lands; the sync page
 *   (B200PROBE_A2A_SYNC_BYTES, zeroed at creation) holds the step-barrier flags of PUSH_SYNC.  A caller
 *   that allocates its own windows must provide 2*world*S + B200PROBE_A2A_SYNC_BYTES bytes and zero the page.
 * create -> (export the 64-byte IPC handle, exchange by any transport, import the peers') ->
 * fill -> exchange.  */
#define B200PROBE_IPC_HANDLE_BYTES 64
#define B200PROBE_A2A_SYNC_BYTES   4096
int b200probe_a2a_window_create(int cuda_ordinal, int world, uint64_t bytes_per_pair,
                                void** window, unsigned char* ipc_handle_out);
int b200probe_a2a_window_fill(int cuda_ordinal, void* window, int rank, int world,
                              uint64_t bytes_per_pair, uint32_t seed, void* stream);
int b200probe_a2a_window_import(int cuda_ordinal, const unsigned char* ipc_handle, void** peer_window);
int b200probe_a2a_window_release(int cuda_ordinal, void* window, int imported);
/* One exchange step of `rank`, asynchronous on `stream`.  windows[r] = base of rank r's window as
 * mapped in THIS process (windows[rank] is the local one).  only_peer: >= 0 that peer only;
 * -1 every slot including the local one; -2 every peer, no local slot (pure NVLink traffic). */
int b200probe_a2a_exchange(int cuda_ordinal, int rank, int world, void* const* windows,
                           uint64_t bytes_per_pair, uint32_t seed, int variant, int ctas_per_peer,
                           int only_peer, void* stream);
/* Seed of the chunk rank `src` sends to rank `dst`. */
uint32_t b200probe_a2a_chunk_seed(uint32_t seed, int src, int dst);

/* ---- tcgen05 GEMM probe (row a13) --------------------------------------------------------------- */
#define B200PROBE_GEMM_OPERANDS_EXACT    0   /* k/128, k integer in [-128,127]: every fp32 partial sum exact -> C bit-exact
                                               against the fp64 contraction rounded once to bf16 (tolerance 0) */
#define B200PROBE_GEMM_OPERANDS_UNIFORM  1   /* SURVEY.md §8d: bf16 U(-1,1) from Philox4x32-10 under key (seed, 0); sampled
                                               outputs within 2^-8 |ref| + 2^-10 sqrt(K) of the fp64 contraction        */
typedef struct b200probe_gemm_cfg {
    int      m, n, k;               /* 0 = 8192; multiples of 128 (256 for the CTA-pair kernel)/256/64 */
    int      warmup, reps;          /* 0,0 = 3,10                                                  */
    uint32_t seed;
    int      samples;               /* sampled outputs checked against fp64 dot products; 0 = 1024 */
    int      operands;              /* B200PROBE_GEMM_OPERANDS_*                                   */
    double   sustain_seconds;       /* >0: additionally run back to back for this long             */
} b200probe_gemm_cfg_t;

typedef struct b200probe_gemm_result {
    int      m, n, k;
    double   ms_median, ms_best;
    double   tflops_median, tflops_best, tflops_sustained;
    double   max_abs_err, max_rel_err;     /* over the sampled outputs, vs fp64                    */
    int      samples, bad;                 /* bad = samples outside tolerance                      */
    uint64_t c_sum64; uint32_t c_xor32;    /* checksum of the bf16 C matrix (run-to-run identity)  */
    int      verified;
    int      operands;                     /* the class that ran                                   */
    double   max_err_over_tol;             /* UNIFORM: max |err| / tolerance over the samples (<= 1) */
} b200probe_gemm_result_t;

/* Operands and C stay resident per device between calls with the same shape, seed and operand class
 * (b200probe_gemm_release frees them; a failed device allocation returns B200PROBE_ENOMEM). */
int b200probe_gemm(int idx, const b200probe_gemm_cfg_t* cfg, b200probe_gemm_result_t* out);
int b200probe_gemm_release(int cuda_ordinal);
/* Resident launch: A [m][k] bf16 row-major, B [n][k] bf16 row-major (i.e. C = A * B^T),
 * C [m][n] bf16.  Asynchronous on stream. */
int b200probe_gemm_launch(int cuda_ordinal, const void* a, const void* b, void* c,
                          int m, int n, int k, void* stream);
/* Deterministic bf16 operand generators used by the probe and restated by the oracle.
 * which: bit 0 = matrix (0 = A, 1 = B), bit 1 = operand class (0 EXACT, 1 UNIFORM), bit 2 = E4M3 (below); dst 16-byte aligned.
 * b200probe_gemm_operand_bits is the same function for one element on the host (the library's own check uses it). */
int b200probe_gemm_fill(int cuda_ordinal, void* dst, uint64_t elems, uint32_t seed, int which, void* stream);
uint16_t b200probe_gemm_operand_bits(uint64_t elem, uint32_t seed, int which);

/* ---- FP8 tensor-core probe (DESIGN.md §4.5): tcgen05.mma kind::f8f6f4, E4M3 x E4M3 -> fp32 -> bf16 --------------------------
 * b200probe_gemm_fill / b200probe_gemm_operand_bits with bit 2 of `which` set generate E4M3 operands, one byte per element
 * (dst receives `elems` bytes; operand_bits returns the byte in the low 8 bits):
 *   EXACT    integers in [-8, 7]: every partial sum is an exact fp32 integer -> C bit-exact against the fp64 contraction
 *            rounded once to bf16
 *   UNIFORM  the UNIFORM class's Philox U(-1,1) fp32 values rounded to E4M3 (nearest even); E4M3 products are exact in
 *            fp32, so the bf16 class's tolerance 2^-8 |ref| + 2^-10 sqrt(K) applies unchanged
 * b200probe_gemm_fp8 takes the same cfg and result as b200probe_gemm, with the same defaults and verdict rules; m and n must
 * be multiples of 256 and k a multiple of 128 (else B200PROBE_EINVAL).  It shares the resident arena that
 * b200probe_gemm_release frees. */
int b200probe_gemm_fp8(int idx, const b200probe_gemm_cfg_t* cfg, b200probe_gemm_result_t* out);
/* Resident launch: A [m][k] and B [n][k] E4M3 row-major (C = A * B^T), C [m][n] bf16, 16-byte aligned.  Asynchronous on stream. */
int b200probe_gemm_fp8_launch(int cuda_ordinal, const void* a, const void* b, void* c,
                              int m, int n, int k, void* stream);

/* ---- data pattern (closed form shared by kernels, oracle and tests) ----------------------------- */
/* word i of a buffer:  ((uint32_t)i * 2654435761u) ^ seed ^ (uint32_t)(i >> 32)                   */
uint32_t b200probe_pattern_word(uint64_t i, uint32_t seed);

#ifdef __cplusplus
}
#endif
#endif /* B200PROBE_H_ */
