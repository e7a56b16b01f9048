// Package b200probe is the cgo binding of libb200probe.so (include/b200probe.h).
//
// NOT COMPILED IN THIS REPOSITORY'S CI: the build image has no Go toolchain (`go version` -> not
// found) and no network to fetch one.  This file is what a maintainer of the NVIDIA
// k8s-device-plugin (installed by /root/reference/README.md:116) would add under internal/ to call
// the probe from the plugin's resource manager; the C++ host (host/cpp) and its Python twin
// (k3s-nvidia_b200/plugin.py) are what runs and is tested here.  See INTEGRATION.md.
package b200probe

/*
#cgo CFLAGS: -I${SRCDIR}/../../../include
#cgo LDFLAGS: -L${SRCDIR}/../../../k3s-nvidia_b200 -lb200probe -Wl,-rpath,${SRCDIR}/../../../k3s-nvidia_b200
#include <stdlib.h>
#include "b200probe.h"
*/
import "C"

import (
	"fmt"
	"runtime"
	"unsafe"
)

// Error carries a b200probe status code (0 OK, <0 library, 1000+cuda, 2000+nvml, 3000+nccl).
type Error struct {
	Code   int
	Detail string
}

func (e *Error) Error() string { return fmt.Sprintf("b200probe: rc=%d (%s)", e.Code, e.Detail) }

func check(rc C.int) error {
	if rc == 0 {
		return nil
	}
	buf := make([]byte, 512)
	C.b200probe_last_error((*C.char)(unsafe.Pointer(&buf[0])), C.int(len(buf)))
	detail := C.GoString((*C.char)(unsafe.Pointer(&buf[0])))
	if detail == "" {
		detail = C.GoString(C.b200probe_strerror(rc))
	}
	return &Error{Code: int(rc), Detail: detail}
}

// Init dlopens NVML (path "" = default) and enumerates. CUDA is initialised lazily by the first probe.
func Init(nvmlPath string) error {
	if nvmlPath == "" {
		return check(C.b200probe_init(nil))
	}
	p := C.CString(nvmlPath)
	defer C.free(unsafe.Pointer(p))
	return check(C.b200probe_init(p))
}

func Shutdown() { C.b200probe_shutdown() }

// Device mirrors b200probe_device_t.
type Device struct {
	Index       int
	UUID, Name  string
	PCIBusID    string
	MemTotal    uint64
	CCMajor     int
	CCMinor     int
	NUMANode    int
	MIGEnabled  int
	CUDAOrdinal int
}

func Devices() ([]Device, error) {
	var n C.int
	if err := check(C.b200probe_device_count(&n)); err != nil {
		return nil, err
	}
	out := make([]Device, 0, int(n))
	for i := 0; i < int(n); i++ {
		var d C.b200probe_device_t
		if err := check(C.b200probe_device_info(C.int(i), &d)); err != nil {
			return nil, err
		}
		out = append(out, Device{
			Index: int(d.index), UUID: C.GoString(&d.uuid[0]), Name: C.GoString(&d.name[0]),
			PCIBusID: C.GoString(&d.pci_bus_id[0]), MemTotal: uint64(d.mem_total),
			CCMajor: int(d.cc_major), CCMinor: int(d.cc_minor), NUMANode: int(d.numa_node),
			MIGEnabled: int(d.mig_enabled), CUDAOrdinal: int(d.cuda_ordinal),
		})
	}
	return out, nil
}

// HealthOpen registers XID/ECC events; disable mirrors env DP_DISABLE_HEALTHCHECKS.
// Returns the bitmask of devices that are Unhealthy from the start.
func HealthOpen(disable string) (uint64, error) {
	p := C.CString(disable)
	defer C.free(unsafe.Pointer(p))
	var m C.uint64_t
	err := check(C.b200probe_health_open(p, &m))
	return uint64(m), err
}

// HealthWait blocks up to timeoutMs in nvmlEventSetWait_v2 and returns the devices that turned
// Unhealthy because of the event (0 on timeout / skipped XID).  Replaces the body of the plugin's
// checkHealth loop: `for { mask, _ := b200probe.HealthWait(5000); for each bit: unhealthy <- d }`.
func HealthWait(timeoutMs int) (newlyUnhealthy uint64, xid uint64, err error) {
	var ev C.b200probe_health_event_t
	err = check(C.b200probe_health_wait(C.int(timeoutMs), &ev))
	return uint64(ev.newly_unhealthy), uint64(ev.event_data), err
}

func HealthClose() { C.b200probe_health_close() }

// HBMPoint mirrors b200probe_hbm_result_t.
type HBMPoint struct {
	Bytes         uint64
	Mode          int
	GBsMedian     float64
	GBsBest       float64
	Sum64         uint64
	Xor32         uint32
	Verified      int
	CacheResident bool
}

// HBMSweep runs the sweep on NVML device idx. CUDA's current device is per OS thread: pin it.
func HBMSweep(idx int, minBytes, maxBytes uint64, modes, warmup, reps int) ([]HBMPoint, error) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	cfg := C.b200probe_hbm_cfg_t{min_bytes: C.uint64_t(minBytes), max_bytes: C.uint64_t(maxBytes), modes: C.int(modes),
		warmup: C.int(warmup), reps: C.int(reps), verify: 1}
	res := make([]C.b200probe_hbm_result_t, 64)
	var n C.int
	err := check(C.b200probe_hbm_sweep(C.int(idx), &cfg, &res[0], C.int(len(res)), &n))
	out := make([]HBMPoint, 0, int(n))
	for i := 0; i < int(n); i++ {
		r := res[i]
		out = append(out, HBMPoint{Bytes: uint64(r.bytes), Mode: int(r.mode), GBsMedian: float64(r.gbs_median),
			GBsBest: float64(r.gbs_best), Sum64: uint64(r.sum64), Xor32: uint32(r.xor32), Verified: int(r.verified),
			CacheResident: r.cache_resident != 0})
	}
	return out, err
}

// NVLinkA2A runs the peer-memory all-to-all over the given CUDA ordinals; pair[i*g+j] = GB/s i->j.
func NVLinkA2A(ordinals []int, bytesPerPair uint64, mode int) (pair []float64, egress []float64, verified bool, err error) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	g := len(ordinals)
	ords := make([]C.int, g)
	for i, o := range ordinals {
		ords[i] = C.int(o)
	}
	cfg := C.b200probe_a2a_cfg_t{bytes_per_pair: C.uint64_t(bytesPerPair), mode: C.int(mode), verify: 1}
	pairC := make([]C.double, g*g)
	var res C.b200probe_a2a_result_t
	err = check(C.b200probe_nvlink_a2a(&ords[0], C.int(g), &cfg, &pairC[0], &res))
	pair = make([]float64, g*g)
	for i := range pair {
		pair[i] = float64(pairC[i])
	}
	egress = make([]float64, g)
	for i := 0; i < g; i++ {
		egress[i] = float64(res.egress_gbs[i])
	}
	// res.pair_source: 0 = shares of a concurrent exchange, 1 = isolated pairs, 2 = drained, device-stamped steps
	return pair, egress, res.verified == 1, err
}

// GEMM runs the tcgen05 probe (0 = 8192 defaults) and returns median TFLOP/s and the data verdict.
// operands: 0 = exact k/128 values (C bit-exact against fp64), 1 = Philox U(-1,1) (sampled outputs within tolerance).
func GEMM(idx, m, n, k, operands int) (tflops float64, verified bool, err error) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	cfg := C.b200probe_gemm_cfg_t{m: C.int(m), n: C.int(n), k: C.int(k), operands: C.int(operands)}
	var res C.b200probe_gemm_result_t
	err = check(C.b200probe_gemm(C.int(idx), &cfg, &res))
	return float64(res.tflops_median), res.verified == 1, err
}

// GEMMFP8 runs the FP8 tensor-core probe (tcgen05.mma kind::f8f6f4, E4M3 operands, bf16 C; 0 = 8192 defaults) and
// returns median TFLOP/s and the data verdict. operands: 0 = integers in [-8, 7] (C bit-exact against fp64), 1 = Philox
// U(-1,1) rounded to E4M3 (sampled outputs within tolerance). m and n must be multiples of 256, k a multiple of 128.
func GEMMFP8(idx, m, n, k, operands int) (tflops float64, verified bool, err error) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	cfg := C.b200probe_gemm_cfg_t{m: C.int(m), n: C.int(n), k: C.int(k), operands: C.int(operands)}
	var res C.b200probe_gemm_result_t
	err = check(C.b200probe_gemm_fp8(C.int(idx), &cfg, &res))
	return float64(res.tflops_median), res.verified == 1, err
}

// GEMMFP8Launch queues one E4M3 GEMM on caller-owned device buffers: A [m][k] and B [n][k] E4M3 row-major, C [m][n]
// bf16, all 16-byte aligned (stream 0 = the default stream).
func GEMMFP8Launch(ordinal int, a, b, c unsafe.Pointer, m, n, k int, stream unsafe.Pointer) error {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	return check(C.b200probe_gemm_fp8_launch(C.int(ordinal), a, b, c, C.int(m), C.int(n), C.int(k), stream))
}

// ErrNoMem is B200PROBE_ENOMEM: a device allocation failed because tenants hold the memory. A resource verdict
// ("inconclusive"), never a health verdict.
const ErrNoMem = -10

// Busy mirrors b200probe_busy_t: who else is on the device (asked before every probe round; busy devices are skipped).
type Busy struct {
	ComputeProcs, UtilGPUPct, UtilMemPct int
	MemUsed                              uint64
	Busy                                 bool
}

func DeviceBusy(idx int) (Busy, error) {
	var b C.b200probe_busy_t
	err := check(C.b200probe_device_busy(C.int(idx), &b))
	return Busy{int(b.compute_procs), int(b.util_gpu_pct), int(b.util_mem_pct), uint64(b.mem_used), b.busy != 0}, err
}

// Release frees every resident probe arena of this process (HBM and GEMM buffers of the listed CUDA ordinals, the
// exchange windows and communicators): called after every probe round so the daemon holds no device memory while tenants run.
func Release(ordinals []int) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	for _, o := range ordinals {
		C.b200probe_hbm_release(C.int(o))
		C.b200probe_gemm_release(C.int(o))
	}
	C.b200probe_a2a_release()
}

// NVLinkStatus mirrors b200probe_nvlink_status_t: the passive NVML view of the links (state per link,
// fabric registration + health mask, DATA/RAW throughput counters) that is correlated with NVLinkA2A.
type NVLinkStatus struct {
	LinksTotal, LinksActive  int
	ActiveMask               uint32
	FabricState, FabricStatus int
	FabricHealthMask         uint32
	DataTxKiB, DataRxKiB     uint64
	RawTxKiB, RawRxKiB       uint64
	CountersOK               bool
}

func NVLinkPassive(idx int) (NVLinkStatus, error) {
	var st C.b200probe_nvlink_status_t
	err := check(C.b200probe_nvlink_passive(C.int(idx), &st))
	return NVLinkStatus{int(st.links_total), int(st.links_active), uint32(st.active_mask), int(st.fabric_state), int(st.fabric_status),
		uint32(st.fabric_health_mask), uint64(st.data_tx_kib), uint64(st.data_rx_kib), uint64(st.raw_tx_kib), uint64(st.raw_rx_kib),
		st.counters_ok == 1}, err
}

// HBMVerify is the probe's verdict pass on a device buffer of CUDA device `ordinal`: checksum of the
// u32 words plus the number of words that differ from the closed-form pattern and the lowest such index.
func HBMVerify(ordinal int, devPtr unsafe.Pointer, bytes uint64, seed uint32) (sum64 uint64, xor32 uint32, bad, first uint64, err error) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	var s, b, f C.uint64_t
	var x C.uint32_t
	err = check(C.b200probe_hbm_verify(C.int(ordinal), devPtr, C.uint64_t(bytes), C.uint32_t(seed), &s, &x, &b, &f))
	return uint64(s), uint32(x), uint64(b), uint64(f), err
}

// ECCStatus mirrors b200probe_ecc_status_t; every field is -1 when NVML cannot report it.
type ECCStatus struct {
	ECCMode                               int
	CorrectedVolatile, UncorrectedVolatile int64
	RemapCorrectedRows, RemapUncorrectedRows int
	RemapPending, RemapFailure            int
}

func eccOf(e *C.b200probe_ecc_status_t) ECCStatus {
	return ECCStatus{int(e.ecc_mode), int64(e.corrected_volatile), int64(e.uncorrected_volatile), int(e.remap_corrected_rows),
		int(e.remap_uncorrected_rows), int(e.remap_pending), int(e.remap_failure)}
}

// HBMECC reads the ECC mode, the volatile corrected / uncorrected totals and the row remapper's state of NVML device idx.
func HBMECC(idx int) (ECCStatus, error) {
	var e C.b200probe_ecc_status_t
	err := check(C.b200probe_hbm_ecc(C.int(idx), &e))
	return eccOf(&e), err
}

// MemtestElement runs one march element on a device buffer of CUDA device `ordinal` (flags: 1 verify, 2 write) and
// returns the mismatching words, the lowest mismatching word index (^0 when none) and the OR of got ^ want.
func MemtestElement(ordinal int, devPtr unsafe.Pointer, bytes, baseWord uint64, flags int, expectSeed, writeSeed uint32) (bad, first uint64, bits uint32, err error) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	var b, f C.uint64_t
	var x C.uint32_t
	err = check(C.b200probe_memtest_element(C.int(ordinal), devPtr, C.uint64_t(bytes), C.uint64_t(baseWord), C.int(flags), C.uint32_t(expectSeed),
		C.uint32_t(writeSeed), &b, &f, &x))
	return uint64(b), uint64(f), uint32(x), err
}

// MemtestResult mirrors b200probe_memtest_result_t.
type MemtestResult struct {
	BytesTested, FreeBefore, Total             uint64
	Chunks, Passes                             int
	AllocMs, TestMs, GBs                       float64
	BadWords, FirstBadWord                     uint64
	BadBits                                    uint32
	FirstBadElement                            int
	ECCCorrectedDelta, ECCUncorrectedDelta     int64
	ECCAfter                                   ECCStatus
}

// HBMMemtest runs the march test over fraction x the free memory of NVML device idx (0 = 0.9) and frees everything
// before it returns. rc -10 (ErrNoMem) = inconclusive: tenants hold the memory.
func HBMMemtest(idx int, fraction float64, passes int) (MemtestResult, error) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	var cfg C.b200probe_memtest_cfg_t
	cfg.fraction = C.double(fraction)
	cfg.passes = C.int(passes)
	var r C.b200probe_memtest_result_t
	err := check(C.b200probe_hbm_memtest(C.int(idx), &cfg, &r))
	return MemtestResult{uint64(r.bytes_tested), uint64(r.free_before), uint64(r.total), int(r.chunks), int(r.passes), float64(r.alloc_ms),
		float64(r.test_ms), float64(r.gbs), uint64(r.bad_words), uint64(r.first_bad_word), uint32(r.bad_bits), int(r.first_bad_element),
		int64(r.ecc_corrected_delta), int64(r.ecc_uncorrected_delta), eccOf(&r.ecc_after)}, err
}

// HostAlloc returns page-locked host memory for HBMCopyHost (C-owned: release with HostFree, never the Go GC).
func HostAlloc(bytes uint64) (unsafe.Pointer, error) {
	var p unsafe.Pointer
	err := check(C.b200probe_host_alloc(C.uint64_t(bytes), &p))
	return p, err
}

func HostFree(p unsafe.Pointer) error { return check(C.b200probe_host_free(p)) }

// HBMCopyHost round-trips src -> device -> dst through the copy kernel (pipelined over chunks) and
// returns the checksum of what landed on the device.  src and dst must be C memory (HostAlloc) or
// pinned Go memory (runtime.Pinner): cgo forbids passing Go pointers that the callee keeps using.
func HBMCopyHost(ordinal int, src, dst unsafe.Pointer, bytes uint64) (sum64 uint64, xor32 uint32, err error) {
	runtime.LockOSThread()
	defer runtime.UnlockOSThread()
	var s C.uint64_t
	var x C.uint32_t
	err = check(C.b200probe_hbm_copy_host(C.int(ordinal), src, dst, C.uint64_t(bytes), &s, &x))
	return uint64(s), uint32(x), err
}
