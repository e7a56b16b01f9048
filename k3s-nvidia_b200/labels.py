"""Probe results -> NFD node labels that gate scheduling (SURVEY.md §5 "NFD label hand-off", §8f.1).

GFD (enabled by /root/reference/values.yaml:1-2) hands labels to Node Feature Discovery by writing
``key=value`` lines into a file under /etc/kubernetes/node-feature-discovery/features.d/; NFD's
*local* source turns them into node labels [RECALLED].  The reference hints at label gating in the
commented selector of /root/reference/nvidia-smi.yaml:6-7 (``nvidia.com/gpu.present: "true"``) and
says the plugin "needs these labels for scheduling" (/root/reference/README.md:99).  We write a
SECOND file in the same directory with ``nvidia.com/b200probe.*`` keys, so no chart value changes.

Thresholds.  north_star asks "healthy at >= 90% of 8 TB/s" (7200 GB/s) and ">= 90% of 900 GB/s/dir".
The driver-measured library copy peak on this pool is 6565.8 GB/s = 82% of 8 TB/s
(MEASURED_PEAKS.json; the part's bus is 7680 bit x 3996 MHz x 2 = 7672 GB/s), so a 7200 GB/s gate
would fail every healthy B200.  Defaults are therefore 90% of the pool-measured healthy figures;
both fractions (of nominal and of measured) are always published, and the north_star gate is one
env var away (B200PROBE_HBM_MIN_GBS=7200).  Once a node has produced one plausible healthy round, its OWN
figures replace the pool constants (calibration file under the state directory).

Tenants.  values.yaml:16-18 time-slices every GPU four ways, so a GPU carrying tenant work is the normal case.
The probes are gated against idle figures and would take SMs, HBM bandwidth and up to 4 GiB per device from
the tenants, so a round first asks NVML who is on each device (b200probe_device_busy) and SKIPS busy devices:
``gpu<i>.probe-state=busy``, the last idle verdict of that GPU is carried over unchanged, and nothing of ours
touches it (B200PROBE_IGNORE_TENANTS=1 turns the check off: benches and tests, where the caller itself is the
tenant).  A failed device allocation (B200PROBE_ENOMEM) is treated the same way (``no-memory``), never as
unhealthy.  (NVML's utilisation figure averages over its last sample period, up to a second: with a probe interval of that order a
round would see the PREVIOUS round's own load and skip — the interval is meant to be minutes, the default is 600 s.)  A GPU that has
never been measured has no verdict and the gate label is absent (selectors on
``...healthy=true`` do not match: unknown is not healthy).  After every round all probe arenas are released.

Staleness.  The file starts with NFD's ``# +expiry-time=`` directive (now + 2 rounds), so a hung or killed daemon
loses its labels; a clean stop removes the file.  There is no timestamp label (it would churn the Node object).
"""
from __future__ import annotations

import logging
import os
import re
import tempfile
import threading
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional

log = logging.getLogger("b200probe.labels")

PREFIX = "nvidia.com/b200probe."
FEATURES_DIR = "/etc/kubernetes/node-feature-discovery/features.d"
FEATURE_FILE = "b200probe"

HBM_NOMINAL_GBS = 8000.0         # north_star's denominator
HBM_MEASURED_GBS = 6565.8        # MEASURED_PEAKS.json hbm_gbs (torch copy_, read+write bytes)
NVLINK_NOMINAL_GBS = 900.0       # per direction per GPU
NVLINK_MEASURED_GBS = 770.0      # /opt/skills/guides/B200_PROFILING.md: peer copy per direction
NVLINK_HEALTHY_GBS = 692.0       # this repo's push kernel with all 18 links up, G = 2 (profiles/a2a_tune_r01_2gpu.txt, +-0.3%)
NVLINK_HEALTHY_GBS_BOX = 700.0   # G > 2: one peer per step with the step barrier (profiles/a2a_sync_relaxed_r01_g8.txt: 701 at every GPU)
GEMM_NOMINAL_TFLOPS = 2250.0
GEMM_MEASURED_TFLOPS = 1670.2
# cuBLASLt FP8 (torch._scaled_mm, E4M3 x E4M3, scales 1.0, bf16 out) at 8192^3, burst median on a B200 at its 1000 W power
# limit, EXACT operands (profiles/gemm_fp8_bench_r01.txt): the pool figure of the FP8 probe until a node has calibrated its own
GEMM_FP8_MEASURED_TFLOPS = 3268.0

_LABEL_VALUE = re.compile(r"^(([A-Za-z0-9][-A-Za-z0-9_.]*)?[A-Za-z0-9])?$")
_LABEL_NAME = re.compile(r"^([A-Za-z0-9][-A-Za-z0-9_.]*)?[A-Za-z0-9]$")


def _env_float(name: str, default: float) -> float:
    try:
        return float(os.environ[name])
    except (KeyError, ValueError):
        return default


@dataclass
class Thresholds:
    hbm_min_gbs: float = field(default_factory=lambda: _env_float("B200PROBE_HBM_MIN_GBS", 0.90 * HBM_MEASURED_GBS))
    # one dead link of 18 costs 5.6% (692 -> ~654 GB/s): the gate sits 3% under the healthy figure for the
    # number of GPUs exchanged (0 = derive from G when the labels are made; B200PROBE_NVLINK_MIN_GBS pins it)
    nvlink_min_gbs: float = field(default_factory=lambda: _env_float("B200PROBE_NVLINK_MIN_GBS", 0.0))
    gemm_min_tflops: float = field(default_factory=lambda: _env_float("B200PROBE_GEMM_MIN_TFLOPS", 0.70 * GEMM_MEASURED_TFLOPS))
    gemm_fp8_min_tflops: float = field(default_factory=lambda: _env_float("B200PROBE_GEMM_FP8_MIN_TFLOPS", 0.70 * GEMM_FP8_MEASURED_TFLOPS))
    verdict_min_bytes: int = 256 << 20        # sizes below L2 are cache-resident: never used for the verdict


def valid_label(key: str, value: str) -> bool:
    if "/" in key:
        pfx, name = key.split("/", 1)
        if len(pfx) > 253:
            return False
    else:
        name = key
    return len(name) <= 63 and bool(_LABEL_NAME.match(name)) and len(value) <= 63 and bool(_LABEL_VALUE.match(value))


def _b(x: bool) -> str:
    return "true" if x else "false"


def hbm_labels(per_gpu: Dict[int, list], th: Thresholds) -> Dict[str, str]:
    """per_gpu: NVML index -> list of HbmPoint.  Verdict = copy GB/s at the largest HBM-resident size."""
    out: Dict[str, str] = {}
    all_ok = True
    worst = None
    for idx, pts in sorted(per_gpu.items()):
        big = [p for p in pts if not p.cache_resident and p.bytes >= th.verdict_min_bytes]
        best = {}
        for mode in ("read", "write", "copy"):
            cand = [p for p in big if p.mode == mode]
            if cand:
                best[mode] = max(cand, key=lambda p: p.bytes)
        data_ok = all(p.verified != 0 for p in pts)
        for mode, p in best.items():
            out[f"{PREFIX}gpu{idx}.hbm-{mode}-gbs"] = str(int(round(p.gbs_median)))
        ok = data_ok and "copy" in best and best["copy"].gbs_median >= th.hbm_min_gbs
        if "copy" in best:
            g = best["copy"].gbs_median
            out[f"{PREFIX}gpu{idx}.hbm-copy-pct-of-nominal"] = str(int(round(100.0 * g / HBM_NOMINAL_GBS)))
            out[f"{PREFIX}gpu{idx}.hbm-copy-pct-of-measured"] = str(int(round(100.0 * g / HBM_MEASURED_GBS)))
            worst = g if worst is None else min(worst, g)
        out[f"{PREFIX}gpu{idx}.hbm-data-ok"] = _b(data_ok)
        out[f"{PREFIX}gpu{idx}.hbm-healthy"] = _b(ok)
        all_ok = all_ok and ok
    out[f"{PREFIX}hbm-healthy"] = _b(all_ok and bool(per_gpu))
    if worst is not None:
        out[f"{PREFIX}hbm-copy-min-gbs"] = str(int(round(worst)))
    return out


def nvlink_labels(rep, th: Thresholds, ids: Optional[List[int]] = None) -> Dict[str, str]:
    """rep: probe.A2aReport.  "Per-link" through NVSwitch means per (src,dst) pair (SURVEY.md §7):
    published per GPU as egress/ingress GB/s plus the cold-spot of the pair matrix.  ids[pos] = the NVML index of the
    GPU at position pos of the exchange (default: position == index)."""
    out: Dict[str, str] = {}
    ok = rep.verified != 0
    ids = list(ids) if ids is not None else list(range(rep.g))
    min_gbs = th.nvlink_min_gbs or (0.97 * NVLINK_HEALTHY_GBS if rep.g <= 2 else 0.96 * NVLINK_HEALTHY_GBS_BOX)
    # G*(G-1) per-pair labels are what BASELINE config 3 asks for ("per-link GB/s surfaced as NFD node labels"); a cluster that
    # only gates on the summary can switch them off (B200PROBE_PAIR_LABELS=0: 56 labels fewer on an 8-GPU node)
    pair_labels = os.environ.get("B200PROBE_PAIR_LABELS", "1") != "0"
    for pos in range(rep.g):
        g = ids[pos]
        out[f"{PREFIX}gpu{g}.nvlink-egress-gbs"] = str(int(round(rep.egress_gbs[pos])))
        out[f"{PREFIX}gpu{g}.nvlink-ingress-gbs"] = str(int(round(rep.ingress_gbs[pos])))
        good = rep.egress_gbs[pos] >= min_gbs
        out[f"{PREFIX}gpu{g}.nvlink-healthy"] = _b(good and rep.verified != 0)
        ok = ok and good
        for q in range(rep.g):
            if pair_labels and q != pos and rep.pair_gbs[pos][q] > 0:
                out[f"{PREFIX}gpu{g}.nvlink-to-gpu{ids[q]}-gbs"] = str(int(round(rep.pair_gbs[pos][q])))
    out[f"{PREFIX}nvlink-min-pair-gbs"] = str(int(round(rep.min_pair_gbs)))
    out[f"{PREFIX}nvlink-egress-pct-of-nominal"] = str(int(round(100.0 * min(rep.egress_gbs[: rep.g]) / NVLINK_NOMINAL_GBS)))
    out[f"{PREFIX}nvlink-data-ok"] = _b(rep.verified != 0)
    out[f"{PREFIX}nvlink-healthy"] = _b(ok)
    return out


def nvlink_passive_labels(per_gpu: Dict[int, dict], expected_links: int = 18) -> Dict[str, str]:
    """per_gpu: NVML index -> Probe.nvlink_passive() dict.  Every link NVML knows must be up and the
    fabric registration completed with a clean health mask (SURVEY.md §8f.3)."""
    out: Dict[str, str] = {}
    all_ok = True
    for idx, st in sorted(per_gpu.items()):
        if st["links_total"] == 0:
            continue                                   # no NVLink on this part: nothing to assert
        ok = st["links_active"] == st["links_total"] and st["links_total"] >= expected_links
        # fabric: a completed registration must have succeeded, and the 2-bit DEGRADED_BW field of the
        # health mask (nvml.h:3453) must not read TRUE (1).  NOT_SUPPORTED / not started is not a fault.
        if st["fabric_state"] == 3 and st["fabric_status"] != 0:
            ok = False
        if (st["fabric_health_mask"] & 0x3) == 1:
            ok = False
        out[f"{PREFIX}gpu{idx}.nvlink-links-active"] = str(st["links_active"])
        out[f"{PREFIX}gpu{idx}.nvlink-links-total"] = str(st["links_total"])
        out[f"{PREFIX}gpu{idx}.nvlink-links-ok"] = _b(ok)
        all_ok = all_ok and ok
    if out:
        out[f"{PREFIX}nvlink-links-ok"] = _b(all_ok)
    return out


def wire_efficiency(before: dict, after: dict):
    """payload / raw bytes on the wire between two passive snapshots (None when the counters are not
    readable): NVML's DATA vs RAW counters quantify the protocol overhead of the active exchange."""
    if not (before.get("counters_ok") and after.get("counters_ok")):
        return None
    d = after["data_tx_kib"] - before["data_tx_kib"]
    r = after["raw_tx_kib"] - before["raw_tx_kib"]
    return (d / r) if r > 0 else None


def gemm_labels(per_gpu: Dict[int, object], th: Thresholds) -> Dict[str, str]:
    out: Dict[str, str] = {}
    all_ok = True
    for idx, r in sorted(per_gpu.items()):
        ok = r.verified == 1 and r.tflops_median >= th.gemm_min_tflops
        out[f"{PREFIX}gpu{idx}.gemm-tflops"] = str(int(round(r.tflops_median)))
        out[f"{PREFIX}gpu{idx}.gemm-data-ok"] = _b(r.verified == 1)
        out[f"{PREFIX}gpu{idx}.gemm-healthy"] = _b(ok)
        all_ok = all_ok and ok
    out[f"{PREFIX}gemm-healthy"] = _b(all_ok and bool(per_gpu))
    return out


def gemm_fp8_labels(per_gpu: Dict[int, object], th: Thresholds) -> Dict[str, str]:
    """The FP8 tensor-core probe (E4M3, tcgen05.mma kind::f8f6f4): the bf16 GEMM's rules on its own keys and threshold."""
    out: Dict[str, str] = {}
    all_ok = True
    for idx, r in sorted(per_gpu.items()):
        ok = r.verified == 1 and r.tflops_median >= th.gemm_fp8_min_tflops
        out[f"{PREFIX}gpu{idx}.gemm-fp8-tflops"] = str(int(round(r.tflops_median)))
        out[f"{PREFIX}gpu{idx}.gemm-fp8-data-ok"] = _b(r.verified == 1)
        out[f"{PREFIX}gpu{idx}.gemm-fp8-healthy"] = _b(ok)
        all_ok = all_ok and ok
    out[f"{PREFIX}gemm-fp8-healthy"] = _b(all_ok and bool(per_gpu))
    return out


def gemm_fp8_enabled() -> bool:
    """B200PROBE_GEMM_FP8=1: every idle GPU also runs the FP8 tensor-core probe; unset or 0 = off."""
    return os.environ.get("B200PROBE_GEMM_FP8", "") not in ("", "0")


def memtest_labels(idx: int, r) -> Dict[str, str]:
    """r: probe.MemtestReport of GPU idx.  The verdict fails on a mismatching word, on uncorrected ECC errors during the
    run and on a failed row remap.  Corrected errors and a pending remap are published only: ECC fixed the data, and a
    pending remap does not affect further work until the next GPU reset applies it (nvml.h:7730)."""
    k = f"{PREFIX}gpu{idx}."
    out = {k + "hbm-memtest-gib": str(int(round(r.bytes_tested / float(1 << 30)))), k + "hbm-memtest-bad-words": str(r.bad_words)}
    if r.ecc_corrected_delta >= 0:
        out[k + "hbm-ecc-corrected-delta"] = str(r.ecc_corrected_delta)
    if r.ecc_uncorrected_delta >= 0:
        out[k + "hbm-ecc-uncorrected-delta"] = str(r.ecc_uncorrected_delta)
    if r.remap_pending >= 0:
        out[k + "hbm-row-remap-pending"] = _b(r.remap_pending == 1)
    if r.remap_failure >= 0:
        out[k + "hbm-row-remap-failed"] = _b(r.remap_failure == 1)
    out[k + "hbm-memtest-healthy"] = _b(r.bad_words == 0 and r.ecc_uncorrected_delta <= 0 and r.remap_failure != 1)
    return out


def memtest_fraction() -> float:
    """B200PROBE_MEMTEST_FRACTION: share of each idle GPU's free memory the march test covers; unset or 0 = off."""
    f = _env_float("B200PROBE_MEMTEST_FRACTION", 0.0)
    return f if 0.0 < f <= 1.0 else 0.0


def gate_label(labels: Dict[str, str]) -> Dict[str, str]:
    """The one label manifests select on: every probe that has a verdict is healthy.  No verdict at all (every GPU
    busy since the daemon started) -> no gate label: unknown is not healthy."""
    parts = [v for k, v in labels.items()
             if k in (f"{PREFIX}hbm-healthy", f"{PREFIX}nvlink-healthy", f"{PREFIX}gemm-healthy", f"{PREFIX}hbm-memtest-healthy",
                      f"{PREFIX}gemm-fp8-healthy")]
    return {f"{PREFIX}healthy": _b(all(v == "true" for v in parts))} if parts else {}


def nvlink_localise(rep, ids: List[int], passive: Dict[int, dict]) -> Dict[str, str]:
    """SURVEY.md §8f.3: join the active pair matrix with the passive per-link state to NAME the suspect.  Through
    NVSwitch every pair sees the same bandwidth, so a cell below 90 % of the matrix's upper quartile is cold; a GPU whose whole
    row (egress) or column (ingress) is cold is the suspect endpoint, and if NVML shows links down on it, those links
    are the evidence.  Only matrices that hold real per-pair rates are used (stepped or isolated, not shares).
    rep.pair_gbs is indexed by position; ids[pos] is the NVML index the labels name."""
    from . import _lib as L

    out: Dict[str, str] = {}
    G = rep.g
    if G < 2 or getattr(rep, "pair_source", L.PAIR_SHARE) == L.PAIR_SHARE:
        return out
    cells = [(rep.pair_gbs[i][j], i, j) for i in range(G) for j in range(G) if i != j and rep.pair_gbs[i][j] > 0]
    if not cells:
        return out
    # healthy reference = the upper quartile of the matrix: one bad endpoint chills 2/G of the cells (half of them at G = 4),
    # so the median can itself be a cold cell; the upper quartile is a healthy cell as long as fewer than 3/4 are cold
    vals = sorted(c[0] for c in cells)
    ref = vals[-((-3 * (len(vals) - 1)) // 4)]
    cold = [(v, i, j) for v, i, j in cells if v < 0.9 * ref]
    out[f"{PREFIX}nvlink-pair-ref-gbs"] = str(int(round(ref)))
    if not cold:
        out[f"{PREFIX}nvlink-cold-cell"] = "none"
        out[f"{PREFIX}nvlink-suspect"] = "none"
        return out
    v, i, j = min(cold)
    out[f"{PREFIX}nvlink-cold-cell"] = f"gpu{ids[i]}-to-gpu{ids[j]}"
    out[f"{PREFIX}nvlink-cold-cells"] = str(len(cold))
    row = [sum(1 for _, a, _b2 in cold if a == g) for g in range(G)]
    col = [sum(1 for _, _a, b2 in cold if b2 == g) for g in range(G)]
    down = {g: passive.get(ids[g], {}) for g in range(G)}
    links_down = [g for g in range(G) if down[g].get("links_total", 0) and down[g].get("links_active", 0) < down[g].get("links_total", 0)]
    # the endpoint with most cold cells; ties go to one that NVML shows links down on
    score = [(row[g] + col[g], g in links_down, -g) for g in range(G)]
    best = max(range(G), key=lambda g: score[g])
    if row[best] + col[best] == 0:
        return out
    out[f"{PREFIX}nvlink-suspect"] = f"gpu{ids[best]}"
    if best in links_down:
        st = down[best]
        mask = ((1 << st["links_total"]) - 1) & ~st["active_mask"]
        out[f"{PREFIX}nvlink-suspect-evidence"] = "links-down"
        out[f"{PREFIX}gpu{ids[best]}.nvlink-links-down-mask"] = f"0x{mask:x}"
    elif G > 2 and row[best] >= (G - 1 + 1) // 2 and col[best] >= (G - 1 + 1) // 2:
        out[f"{PREFIX}nvlink-suspect-evidence"] = "port-both-directions"
    elif G > 2 and row[best] > col[best] and row[best] >= 2:
        out[f"{PREFIX}nvlink-suspect-evidence"] = "egress-cold"
    elif G > 2 and col[best] > row[best] and col[best] >= 2:
        out[f"{PREFIX}nvlink-suspect-evidence"] = "ingress-cold"
    else:
        out[f"{PREFIX}nvlink-suspect-evidence"] = "pair-only"
    return out


def render(labels: Dict[str, str], expiry_unix: Optional[float] = None) -> str:
    bad = [(k, v) for k, v in labels.items() if not valid_label(k, v)]
    if bad:
        raise ValueError(f"invalid label(s): {bad}")
    head = ""
    if expiry_unix is not None:      # NFD local source [RECALLED, NFD >= 0.14]: labels of this file are dropped after this instant
        head = "# +expiry-time=" + time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime(expiry_unix)) + "\n"
    return head + "".join(f"{k}={v}\n" for k, v in sorted(labels.items()))


def write_feature_file(labels: Dict[str, str], features_dir: str = FEATURES_DIR, name: str = FEATURE_FILE, expiry_unix: Optional[float] = None) -> str:
    """Atomic replace (NFD may read at any time): write a hidden temp file, then rename."""
    os.makedirs(features_dir, exist_ok=True)
    text = render(labels, expiry_unix)
    fd, tmp = tempfile.mkstemp(prefix=".", suffix=".tmp", dir=features_dir)   # dot-files are ignored by NFD
    try:
        with os.fdopen(fd, "w") as f:
            f.write(text)
        os.chmod(tmp, 0o644)
        path = os.path.join(features_dir, name)
        os.replace(tmp, path)
    finally:
        if os.path.exists(tmp):
            os.unlink(tmp)
    return path


def parse_feature_file(text: str) -> Dict[str, str]:
    out = {}
    for line in text.splitlines():
        line = line.strip()
        if not line or line.startswith("#"):
            continue
        k, _, v = line.partition("=")
        out[k] = v
    return out


_GPU_KEY = re.compile(r"^" + re.escape(PREFIX) + r"gpu(\d+)\.(.+)$")
ENOMEM = -10          # B200PROBE_ENOMEM


class Calibration:
    """This node's own healthy figures (first plausible healthy round), kept as key=value lines under the state
    directory.  A figure is accepted once, when its data check passed and it is within 15 % of the pool figure, and
    from then on the gate is a fraction of THAT instead of the pool constant."""

    def __init__(self, state_dir: str):
        self.path = os.path.join(state_dir, "calibration")
        self.vals: Dict[str, float] = {}
        try:
            with open(self.path) as f:
                for k, v in parse_feature_file(f.read()).items():
                    self.vals[k] = float(v)
        except (OSError, ValueError):
            pass

    def get(self, key: str, pool: float) -> float:
        return self.vals.get(key, pool)

    def offer(self, key: str, value: float, pool: float) -> None:
        if key not in self.vals and 0.85 * pool <= value <= 1.15 * pool:
            self.vals[key] = value
            os.makedirs(os.path.dirname(self.path), exist_ok=True)
            tmp = self.path + ".tmp"
            with open(tmp, "w") as f:
                f.write("".join(f"{k}={v:.1f}\n" for k, v in sorted(self.vals.items())))
            os.replace(tmp, self.path)


class ActiveProbeRunner:
    """Runs the active probes on every enumerated, IDLE GPU at an interval and publishes the labels.  A probe that fails
    for a reason of the GPU (CUDA error, data mismatch, too slow) publishes ``…healthy=false``; a GPU that is in use or
    has no memory to spare is skipped and keeps its last idle verdict.  Never blocks ListAndWatch (separate thread,
    separate CUDA streams); holds no device memory between rounds."""

    def __init__(self, probe, *, features_dir: str = FEATURES_DIR, interval_s: float = 600.0, thresholds: Optional[Thresholds] = None,
                 hbm_kwargs: Optional[dict] = None, run_nvlink: bool = True, run_gemm: bool = True, keep_arenas: bool = False,
                 state_dir: Optional[str] = None):
        self.probe = probe
        self.features_dir = features_dir
        self.interval_s = interval_s
        self.th = thresholds or Thresholds()
        self._explicit_hbm_gate = thresholds is not None or "B200PROBE_HBM_MIN_GBS" in os.environ
        self._explicit_gemm_gate = thresholds is not None or "B200PROBE_GEMM_MIN_TFLOPS" in os.environ
        self._explicit_gemm_fp8_gate = thresholds is not None or "B200PROBE_GEMM_FP8_MIN_TFLOPS" in os.environ
        self.hbm_kwargs = hbm_kwargs or dict(min_bytes=1 << 28, max_bytes=1 << 30, warmup=2, reps=5, verify=1)
        self.run_nvlink = run_nvlink
        self.run_gemm = run_gemm
        self.keep_arenas = keep_arenas
        self.cal = Calibration(state_dir or os.environ.get("B200PROBE_STATE_DIR") or os.path.join(features_dir, ".b200probe-state"))
        self._stop = threading.Event()
        self._thread: Optional[threading.Thread] = None
        self.last_labels: Dict[str, str] = {}
        self.last_round_s = 0.0

    # -- helpers -----------------------------------------------------------------------------------
    def _carry(self, labels: Dict[str, str], idx: int, leaf_prefix: str) -> None:
        """A skipped GPU keeps the per-GPU labels of its last measured round."""
        for k, v in self.last_labels.items():
            m = _GPU_KEY.match(k)
            if m and int(m.group(1)) == idx and m.group(2).startswith(leaf_prefix) and k not in labels:
                labels[k] = v

    @staticmethod
    def _aggregate(labels: Dict[str, str], leaf: str) -> None:
        vals = [v for k, v in labels.items() if (m := _GPU_KEY.match(k)) and m.group(2) == leaf]
        if vals:
            labels[f"{PREFIX}{leaf}"] = _b(all(v == "true" for v in vals))
        else:
            labels.pop(f"{PREFIX}{leaf}", None)

    def release(self) -> None:
        """Free every probe arena of this process (device memory, streams, NCCL communicators)."""
        ords = [d.cuda_ordinal for d in (self.probe.device_info(i) for i in range(self.probe.device_count())) if d.cuda_ordinal >= 0]
        self.probe.release(ords)

    def run_once(self) -> Dict[str, str]:
        from .probe import ProbeError

        t_round = time.perf_counter()
        labels: Dict[str, str] = {}
        n = self.probe.device_count()
        infos = [self.probe.device_info(i) for i in range(n)]
        # who is on the devices?  asked once, before any probe of ours shows up in the utilisation figures
        state: Dict[int, str] = {}
        ignore_tenants = os.environ.get("B200PROBE_IGNORE_TENANTS", "") not in ("", "0")      # benches / tests: the caller IS the tenant
        for d in infos:
            try:
                state[d.index] = "busy" if (not ignore_tenants and self.probe.device_busy(d.index)["busy"]) else "probed"
            except Exception as e:  # noqa: BLE001
                log.warning("busy query failed on GPU %d (%s): probing it", d.index, e)
                state[d.index] = "probed"
        hbm, gemm = {}, {}
        for d in infos:
            if state[d.index] != "probed":
                continue
            try:
                hbm[d.index] = self.probe.hbm_sweep(d.index, **self.hbm_kwargs)
            except ProbeError as e:
                if e.rc == ENOMEM:
                    state[d.index] = "no-memory"
                    log.warning("GPU %d: no device memory for the HBM probe (tenants hold it): inconclusive", d.index)
                    continue
                log.error("HBM probe failed on GPU %d: %s", d.index, e)
                labels[f"{PREFIX}gpu{d.index}.hbm-healthy"] = "false"
            except Exception as e:  # noqa: BLE001
                log.error("HBM probe failed on GPU %d: %s", d.index, e)
                labels[f"{PREFIX}gpu{d.index}.hbm-healthy"] = "false"
        for idx, pts in sorted(hbm.items()):
            uuid = infos[idx].uuid
            th = self.th
            if not self._explicit_hbm_gate:
                th = Thresholds(hbm_min_gbs=0.90 * self.cal.get(f"hbm-copy-gbs.{uuid}", HBM_MEASURED_GBS), nvlink_min_gbs=self.th.nvlink_min_gbs,
                                gemm_min_tflops=self.th.gemm_min_tflops)
            got = hbm_labels({idx: pts}, th)
            labels.update({k: v for k, v in got.items() if _GPU_KEY.match(k)})
            if got.get(f"{PREFIX}gpu{idx}.hbm-healthy") == "true" and f"{PREFIX}gpu{idx}.hbm-copy-gbs" in got:
                self.cal.offer(f"hbm-copy-gbs.{uuid}", float(got[f"{PREFIX}gpu{idx}.hbm-copy-gbs"]), HBM_MEASURED_GBS)
        if self.run_gemm:
            for d in infos:
                if state[d.index] != "probed":
                    continue
                try:
                    gemm[d.index] = self.probe.gemm(d.index, warmup=2, reps=5)
                except ProbeError as e:
                    if e.rc == ENOMEM:
                        state[d.index] = "no-memory"
                        continue
                    log.error("GEMM probe failed on GPU %d: %s", d.index, e)
                    labels[f"{PREFIX}gpu{d.index}.gemm-healthy"] = "false"
                except Exception as e:  # noqa: BLE001
                    log.error("GEMM probe failed on GPU %d: %s", d.index, e)
                    labels[f"{PREFIX}gpu{d.index}.gemm-healthy"] = "false"
            for idx, r in sorted(gemm.items()):
                uuid = infos[idx].uuid
                th = self.th
                if not self._explicit_gemm_gate:
                    th = Thresholds(hbm_min_gbs=self.th.hbm_min_gbs, nvlink_min_gbs=self.th.nvlink_min_gbs,
                                    gemm_min_tflops=0.70 * self.cal.get(f"gemm-tflops.{uuid}", GEMM_MEASURED_TFLOPS))
                got = gemm_labels({idx: r}, th)
                labels.update({k: v for k, v in got.items() if _GPU_KEY.match(k)})
                if got.get(f"{PREFIX}gpu{idx}.gemm-healthy") == "true":
                    self.cal.offer(f"gemm-tflops.{uuid}", r.tflops_median, GEMM_MEASURED_TFLOPS)
        if gemm_fp8_enabled():
            for d in infos:
                if state[d.index] != "probed":
                    continue
                try:
                    r = self.probe.gemm_fp8(d.index, warmup=2, reps=5)
                except ProbeError as e:
                    if e.rc == ENOMEM:
                        state[d.index] = "no-memory"
                        log.warning("GPU %d: no device memory for the FP8 GEMM probe (tenants hold it): inconclusive", d.index)
                        continue
                    log.error("FP8 GEMM probe failed on GPU %d: %s", d.index, e)
                    labels[f"{PREFIX}gpu{d.index}.gemm-fp8-healthy"] = "false"
                    continue
                except Exception as e:  # noqa: BLE001
                    log.error("FP8 GEMM probe failed on GPU %d: %s", d.index, e)
                    labels[f"{PREFIX}gpu{d.index}.gemm-fp8-healthy"] = "false"
                    continue
                uuid = infos[d.index].uuid
                th = self.th
                if not self._explicit_gemm_fp8_gate:
                    th = Thresholds(hbm_min_gbs=self.th.hbm_min_gbs, nvlink_min_gbs=self.th.nvlink_min_gbs, gemm_min_tflops=self.th.gemm_min_tflops,
                                    gemm_fp8_min_tflops=0.70 * self.cal.get(f"gemm-fp8-tflops.{uuid}", GEMM_FP8_MEASURED_TFLOPS))
                got = gemm_fp8_labels({d.index: r}, th)
                labels.update({k: v for k, v in got.items() if _GPU_KEY.match(k)})
                if got.get(f"{PREFIX}gpu{d.index}.gemm-fp8-healthy") == "true":
                    self.cal.offer(f"gemm-fp8-tflops.{uuid}", r.tflops_median, GEMM_FP8_MEASURED_TFLOPS)
        fraction = memtest_fraction()
        if fraction > 0:
            for d in infos:
                if state[d.index] != "probed":
                    continue
                try:
                    labels.update(memtest_labels(d.index, self.probe.hbm_memtest(d.index, fraction=fraction)))
                except ProbeError as e:
                    if e.rc == ENOMEM:
                        state[d.index] = "no-memory"
                        log.warning("GPU %d: no device memory for the HBM memtest (tenants hold it): inconclusive", d.index)
                        continue
                    log.error("HBM memtest failed on GPU %d: %s", d.index, e)
                    labels[f"{PREFIX}gpu{d.index}.hbm-memtest-healthy"] = "false"
                except Exception as e:  # noqa: BLE001
                    log.error("HBM memtest failed on GPU %d: %s", d.index, e)
                    labels[f"{PREFIX}gpu{d.index}.hbm-memtest-healthy"] = "false"
        # GPUs that were skipped keep what their last measured round said
        for d in infos:
            labels[f"{PREFIX}gpu{d.index}.probe-state"] = state[d.index]
            if state[d.index] != "probed":
                self._carry(labels, d.index, "hbm-")
                self._carry(labels, d.index, "gemm-")
        self._aggregate(labels, "hbm-healthy")
        self._aggregate(labels, "hbm-memtest-healthy")
        self._aggregate(labels, "gemm-fp8-healthy")
        if self.run_gemm:
            self._aggregate(labels, "gemm-healthy")
        copies = [float(v) for k, v in labels.items() if (m := _GPU_KEY.match(k)) and m.group(2) == "hbm-copy-gbs"]
        if copies:
            labels[f"{PREFIX}hbm-copy-min-gbs"] = str(int(round(min(copies))))

        # ---- NVLink: passive state of every GPU, the exchange over the idle ones -----------------------------------
        passive_before = {}
        try:
            passive_before = {d.index: self.probe.nvlink_passive(d.index) for d in infos}
            labels.update(nvlink_passive_labels(passive_before))
        except Exception as e:  # noqa: BLE001
            log.error("passive NVLink status failed: %s", e)
        # re-read the devices: CUDA ordinals are resolved (by UUID) by the first probe call of the process, not at enumeration
        idle = [d for d in (self.probe.device_info(i) for i in range(n)) if state[d.index] == "probed" and d.cuda_ordinal >= 0]
        ran_nvlink = False
        if self.run_nvlink and len(idle) >= 2:
            ids = [d.index for d in idle]
            try:
                rep = self.probe.nvlink_a2a([d.cuda_ordinal for d in idle], warmup=2, reps=5)
                labels.update(nvlink_labels(rep, self.th, ids))
                labels.update(nvlink_localise(rep, ids, passive_before))
                if labels.get(f"{PREFIX}nvlink-links-ok") == "false":
                    labels[f"{PREFIX}nvlink-healthy"] = "false"      # a dead link fails the gate even if the matrix still clears the bar
                eff = [wire_efficiency(passive_before[i], self.probe.nvlink_passive(i)) for i in ids if i in passive_before]
                eff = [e for e in eff if e]
                if eff:
                    labels[f"{PREFIX}nvlink-data-over-raw-pct"] = str(int(round(100.0 * min(eff))))
                ran_nvlink = True
            except ProbeError as e:
                if e.rc == ENOMEM:
                    log.warning("no device memory for the NVLink exchange: inconclusive")
                else:
                    log.error("NVLink probe failed: %s", e)
                    labels[f"{PREFIX}nvlink-healthy"] = "false"
                    ran_nvlink = True
            except Exception as e:  # noqa: BLE001
                log.error("NVLink probe failed: %s", e)
                labels[f"{PREFIX}nvlink-healthy"] = "false"
                ran_nvlink = True
        if self.run_nvlink and not ran_nvlink:
            # nothing measured this round (GPUs busy / a single GPU): the whole NVLink picture of the last measured round stands
            for k, v in self.last_labels.items():
                if "nvlink-" in k and "nvlink-links-" not in k and k not in labels:
                    labels[k] = v
        labels.update(gate_label(labels))
        if not self.keep_arenas:
            try:
                self.release()
            except Exception as e:  # noqa: BLE001
                log.warning("releasing probe arenas failed: %s", e)
        self.last_labels = labels
        self.last_round_s = time.perf_counter() - t_round
        log.info("active probe round: %.2f s, gate=%s, states=%s", self.last_round_s, labels.get(f"{PREFIX}healthy", "absent"), state)
        write_feature_file(labels, self.features_dir, expiry_unix=time.time() + 2.0 * self.interval_s + 60.0)
        return labels

    def withdraw(self) -> None:
        """Clean shutdown: the verdicts are no longer maintained, so they are removed (NFD drops the labels)."""
        try:
            os.unlink(os.path.join(self.features_dir, FEATURE_FILE))
        except OSError:
            pass

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.run_once()
            except Exception as e:  # noqa: BLE001
                log.error("active probe round failed: %s", e)
            self._stop.wait(self.interval_s)

    def start(self):
        self._thread = threading.Thread(target=self._loop, name="b200probe-active", daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=5.0)
        self.withdraw()
