// Probe results -> NFD node labels that gate scheduling (SURVEY.md §5 "NFD label hand-off", §8f.1).
// Native twin of k3s-nvidia_b200/labels.py: same keys, same rounding, same thresholds, same file format.
//
// GFD (enabled by /root/reference/values.yaml:1-2) hands labels to Node Feature Discovery by writing
// key=value lines into a file under /etc/kubernetes/node-feature-discovery/features.d/ [RECALLED]; the
// reference hints at label gating in the commented selector of /root/reference/nvidia-smi.yaml:6-7 and says
// the plugin "needs these labels for scheduling" (/root/reference/README.md:99).  We write a SECOND file in
// the same directory with nvidia.com/b200probe.* keys, so no chart value changes.
//
// Tenants (values.yaml:16-18 time-slices every GPU four ways): a round first asks NVML who is on each device
// (b200probe_device_busy) and SKIPS busy devices — probe-state=busy, the last idle verdict carried over, nothing of ours
// touches the device; a failed device allocation (B200PROBE_ENOMEM) is handled the same way (no-memory), never as
// unhealthy.  A GPU never measured has no verdict and the gate label is absent.  All probe arenas are released after
// every round.  The file carries NFD's "# +expiry-time=" directive (now + 2 rounds) and is removed on a clean stop;
// there is no timestamp label.  Gates follow this node's own first plausible healthy figures (calibration file).
#pragma once
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <ctime>
#include <fstream>
#include <map>
#include <set>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b200probe.h"
#include "plugin.hpp"

namespace labels {

static const char kPrefix[] = "nvidia.com/b200probe.";
static const double kHbmNominal = 8000.0, kHbmMeasured = 6565.8;            // north_star's denominator; MEASURED_PEAKS.json hbm_gbs
static const double kNvlinkNominal = 900.0;
static const double kNvlinkHealthyPair = 692.0, kNvlinkHealthyBox = 700.0;  // profiles/a2a_tune_r01_2gpu.txt; profiles/a2a_sync_relaxed_r01_g8.txt
static const double kGemmMeasured = 1670.2;
// cuBLASLt FP8 (torch._scaled_mm, E4M3 x E4M3, scales 1.0, bf16 out) at 8192^3, burst median on a B200 at its 1000 W power
// limit, EXACT operands (profiles/gemm_fp8_bench_r01.txt); twin of labels.py GEMM_FP8_MEASURED_TFLOPS
static const double kGemmFp8Measured = 3268.0;

using Labels = std::map<std::string, std::string>;

inline double env_double(const char* name, double dflt) {
    const char* e = getenv(name);
    if (!e || !*e) return dflt;
    char* end = nullptr;
    const double v = strtod(e, &end);
    return (end && *end == 0) ? v : dflt;
}

struct Thresholds {
    double hbm_min_gbs = env_double("B200PROBE_HBM_MIN_GBS", 0.90 * kHbmMeasured);
    double nvlink_min_gbs = env_double("B200PROBE_NVLINK_MIN_GBS", 0.0);     // 0 = 97 % of the healthy figure for the number of GPUs exchanged
    double gemm_min_tflops = env_double("B200PROBE_GEMM_MIN_TFLOPS", 0.70 * kGemmMeasured);
    double gemm_fp8_min_tflops = env_double("B200PROBE_GEMM_FP8_MIN_TFLOPS", 0.70 * kGemmFp8Measured);
    uint64_t verdict_min_bytes = 256ull << 20;                                // sizes below L2 are cache-resident: never used for the verdict
};

inline std::string b(bool x) { return x ? "true" : "false"; }
// Python's round(): half to even
inline std::string rint_str(double v) { return std::to_string((long long)std::nearbyint(v)); }
inline std::string key(int gpu, const char* leaf) { return std::string(kPrefix) + "gpu" + std::to_string(gpu) + "." + leaf; }
inline std::string key(const char* leaf) { return std::string(kPrefix) + leaf; }

inline bool valid_label(const std::string& k, const std::string& v) {
    auto name_ok = [](const std::string& s, bool allow_empty) {
        if (s.empty()) return allow_empty;
        if (s.size() > 63 || !isalnum((unsigned char)s.front()) || !isalnum((unsigned char)s.back())) return false;
        for (unsigned char c : s) if (!isalnum(c) && c != '-' && c != '_' && c != '.') return false;
        return true;
    };
    std::string name = k;
    const size_t slash = k.find('/');
    if (slash != std::string::npos) { if (slash > 253) return false; name = k.substr(slash + 1); }
    return name_ok(name, false) && name_ok(v, true);
}

inline Labels hbm_labels(const std::map<int, std::vector<b200probe_hbm_result_t>>& per_gpu, const Thresholds& th) {
    Labels out;
    bool all_ok = true, have_worst = false;
    double worst = 0;
    for (const auto& kv : per_gpu) {
        const int idx = kv.first;
        const b200probe_hbm_result_t* best[3] = {nullptr, nullptr, nullptr};   // read, write, copy at the largest HBM-resident size
        static const int modes[3] = {B200PROBE_HBM_READ, B200PROBE_HBM_WRITE, B200PROBE_HBM_COPY};
        static const char* names[3] = {"read", "write", "copy"};
        bool data_ok = true;
        for (const auto& p : kv.second) {
            if (p.verified == 0) data_ok = false;
            if (p.cache_resident || p.bytes < th.verdict_min_bytes) continue;
            for (int m = 0; m < 3; ++m) if (p.mode == modes[m] && (!best[m] || p.bytes > best[m]->bytes)) best[m] = &p;
        }
        for (int m = 0; m < 3; ++m) if (best[m]) out[key(idx, (std::string("hbm-") + names[m] + "-gbs").c_str())] = rint_str(best[m]->gbs_median);
        const bool ok = data_ok && best[2] && best[2]->gbs_median >= th.hbm_min_gbs;
        if (best[2]) {
            const double g = best[2]->gbs_median;
            out[key(idx, "hbm-copy-pct-of-nominal")] = rint_str(100.0 * g / kHbmNominal);
            out[key(idx, "hbm-copy-pct-of-measured")] = rint_str(100.0 * g / kHbmMeasured);
            worst = have_worst ? std::min(worst, g) : g;
            have_worst = true;
        }
        out[key(idx, "hbm-data-ok")] = b(data_ok);
        out[key(idx, "hbm-healthy")] = b(ok);
        all_ok = all_ok && ok;
    }
    out[key("hbm-healthy")] = b(all_ok && !per_gpu.empty());
    if (have_worst) out[key("hbm-copy-min-gbs")] = rint_str(worst);
    return out;
}

// ids[pos] = NVML index of the GPU at position pos of the exchange (the labels name NVML indices)
inline Labels nvlink_labels(const b200probe_a2a_result_t& rep, const std::vector<double>& pair_gbs, const Thresholds& th, std::vector<int> ids = {}) {
    Labels out;
    const int G = rep.g;
    if (ids.empty()) for (int i = 0; i < G; ++i) ids.push_back(i);
    bool ok = rep.verified != 0;
    const double min_gbs = th.nvlink_min_gbs > 0 ? th.nvlink_min_gbs : (G <= 2 ? 0.97 * kNvlinkHealthyPair : 0.96 * kNvlinkHealthyBox);
    double min_egress = 1e300;
    const char* pl = getenv("B200PROBE_PAIR_LABELS");                 // "0": no per-pair labels (the summary and the localisation stay)
    const bool pair_labels = !(pl && strcmp(pl, "0") == 0);
    for (int pos = 0; pos < G; ++pos) {
        const int g = ids[(size_t)pos];
        out[key(g, "nvlink-egress-gbs")] = rint_str(rep.egress_gbs[pos]);
        out[key(g, "nvlink-ingress-gbs")] = rint_str(rep.ingress_gbs[pos]);
        const bool good = rep.egress_gbs[pos] >= min_gbs;
        out[key(g, "nvlink-healthy")] = b(good && rep.verified != 0);
        ok = ok && good;
        min_egress = std::min(min_egress, rep.egress_gbs[pos]);
        for (int q = 0; q < G; ++q)
            if (pair_labels && q != pos && pair_gbs[(size_t)(pos * G + q)] > 0)
                out[key(g, ("nvlink-to-gpu" + std::to_string(ids[(size_t)q]) + "-gbs").c_str())] = rint_str(pair_gbs[(size_t)(pos * G + q)]);
    }
    out[key("nvlink-min-pair-gbs")] = rint_str(rep.min_pair_gbs);
    out[key("nvlink-egress-pct-of-nominal")] = rint_str(100.0 * min_egress / kNvlinkNominal);
    out[key("nvlink-data-ok")] = b(rep.verified != 0);
    out[key("nvlink-healthy")] = b(ok);
    return out;
}

// Every link NVML knows must be up and the fabric registration completed with a clean health mask (§8f.3).
inline Labels nvlink_passive_labels(const std::map<int, b200probe_nvlink_status_t>& per_gpu, int expected_links = 18) {
    Labels out;
    bool all_ok = true;
    for (const auto& kv : per_gpu) {
        const auto& st = kv.second;
        if (st.links_total == 0) continue;                         // no NVLink on this part: nothing to assert
        bool ok = st.links_active == st.links_total && st.links_total >= expected_links;
        if (st.fabric_state == 3 && st.fabric_status != 0) ok = false;
        if ((st.fabric_health_mask & 0x3) == 1) ok = false;        // DEGRADED_BW == TRUE (nvml.h:3453)
        out[key(kv.first, "nvlink-links-active")] = std::to_string(st.links_active);
        out[key(kv.first, "nvlink-links-total")] = std::to_string(st.links_total);
        out[key(kv.first, "nvlink-links-ok")] = b(ok);
        all_ok = all_ok && ok;
    }
    if (!out.empty()) out[key("nvlink-links-ok")] = b(all_ok);
    return out;
}

inline Labels gemm_labels(const std::map<int, b200probe_gemm_result_t>& per_gpu, const Thresholds& th) {
    Labels out;
    bool all_ok = true;
    for (const auto& kv : per_gpu) {
        const auto& r = kv.second;
        const bool ok = r.verified == 1 && r.tflops_median >= th.gemm_min_tflops;
        out[key(kv.first, "gemm-tflops")] = rint_str(r.tflops_median);
        out[key(kv.first, "gemm-data-ok")] = b(r.verified == 1);
        out[key(kv.first, "gemm-healthy")] = b(ok);
        all_ok = all_ok && ok;
    }
    out[key("gemm-healthy")] = b(all_ok && !per_gpu.empty());
    return out;
}

// Twin of labels.py gemm_fp8_labels: the bf16 GEMM's rules on the FP8 probe's own keys and threshold
inline Labels gemm_fp8_labels(const std::map<int, b200probe_gemm_result_t>& per_gpu, const Thresholds& th) {
    Labels out;
    bool all_ok = true;
    for (const auto& kv : per_gpu) {
        const auto& r = kv.second;
        const bool ok = r.verified == 1 && r.tflops_median >= th.gemm_fp8_min_tflops;
        out[key(kv.first, "gemm-fp8-tflops")] = rint_str(r.tflops_median);
        out[key(kv.first, "gemm-fp8-data-ok")] = b(r.verified == 1);
        out[key(kv.first, "gemm-fp8-healthy")] = b(ok);
        all_ok = all_ok && ok;
    }
    out[key("gemm-fp8-healthy")] = b(all_ok && !per_gpu.empty());
    return out;
}

// B200PROBE_GEMM_FP8=1: every idle GPU also runs the FP8 tensor-core probe; unset or 0 = off
inline bool gemm_fp8_enabled() {
    const char* e = getenv("B200PROBE_GEMM_FP8");
    return e && *e && strcmp(e, "0") != 0;
}

// Twin of labels.py memtest_labels: a mismatching word, uncorrected ECC errors during the run or a failed row remap fail
// the verdict; corrected errors and a pending remap are published only (a pending remap does not affect further work).
inline Labels memtest_labels(int idx, const b200probe_memtest_result_t& r) {
    Labels out;
    out[key(idx, "hbm-memtest-gib")] = rint_str((double)r.bytes_tested / (double)(1ull << 30));
    out[key(idx, "hbm-memtest-bad-words")] = std::to_string((unsigned long long)r.bad_words);
    if (r.ecc_corrected_delta >= 0) out[key(idx, "hbm-ecc-corrected-delta")] = std::to_string((long long)r.ecc_corrected_delta);
    if (r.ecc_uncorrected_delta >= 0) out[key(idx, "hbm-ecc-uncorrected-delta")] = std::to_string((long long)r.ecc_uncorrected_delta);
    if (r.ecc_after.remap_pending >= 0) out[key(idx, "hbm-row-remap-pending")] = b(r.ecc_after.remap_pending == 1);
    if (r.ecc_after.remap_failure >= 0) out[key(idx, "hbm-row-remap-failed")] = b(r.ecc_after.remap_failure == 1);
    out[key(idx, "hbm-memtest-healthy")] = b(r.bad_words == 0 && r.ecc_uncorrected_delta <= 0 && r.ecc_after.remap_failure != 1);
    return out;
}

// B200PROBE_MEMTEST_FRACTION: share of each idle GPU's free memory the march test covers; unset or 0 = off
inline double memtest_fraction() {
    const double f = env_double("B200PROBE_MEMTEST_FRACTION", 0.0);
    return f > 0.0 && f <= 1.0 ? f : 0.0;
}

// The one label manifests select on: every probe that has a verdict is healthy.  No verdict at all -> no gate label.
inline void gate_label(Labels* l) {
    bool any = false, all = true;
    for (const char* leaf : {"hbm-healthy", "nvlink-healthy", "gemm-healthy", "hbm-memtest-healthy", "gemm-fp8-healthy"}) {
        auto it = l->find(key(leaf));
        if (it != l->end()) { any = true; all = all && it->second == "true"; }
    }
    if (any) (*l)[key("healthy")] = b(all);
}

// SURVEY.md §8f.3: join the active pair matrix with the passive per-link state to NAME the suspect (twin of
// labels.py nvlink_localise: same reference = upper quartile of the matrix, same 90 % cold bar, same tie-breaks).
inline Labels nvlink_localise(const b200probe_a2a_result_t& rep, const std::vector<double>& pair, const std::vector<int>& ids,
                              const std::map<int, b200probe_nvlink_status_t>& passive) {
    Labels out;
    const int G = rep.g;
    if (G < 2 || rep.pair_source == B200PROBE_PAIR_SHARE) return out;
    struct Cell { double v; int i, j; };
    std::vector<Cell> cells;
    for (int i = 0; i < G; ++i) for (int j = 0; j < G; ++j) if (i != j && pair[(size_t)(i * G + j)] > 0) cells.push_back({pair[(size_t)(i * G + j)], i, j});
    if (cells.empty()) return out;
    std::vector<double> vals;
    for (const auto& c : cells) vals.push_back(c.v);
    std::sort(vals.begin(), vals.end());
    const double ref = vals[(3 * (vals.size() - 1) + 3) / 4];
    out[key("nvlink-pair-ref-gbs")] = rint_str(ref);
    std::vector<Cell> cold;
    for (const auto& c : cells) if (c.v < 0.9 * ref) cold.push_back(c);
    if (cold.empty()) { out[key("nvlink-cold-cell")] = "none"; out[key("nvlink-suspect")] = "none"; return out; }
    const Cell* worst = &cold[0];
    for (const auto& c : cold) if (c.v < worst->v || (c.v == worst->v && (c.i < worst->i || (c.i == worst->i && c.j < worst->j)))) worst = &c;
    out[key("nvlink-cold-cell")] = "gpu" + std::to_string(ids[(size_t)worst->i]) + "-to-gpu" + std::to_string(ids[(size_t)worst->j]);
    out[key("nvlink-cold-cells")] = std::to_string(cold.size());
    std::vector<int> row((size_t)G, 0), col((size_t)G, 0);
    for (const auto& c : cold) { row[(size_t)c.i]++; col[(size_t)c.j]++; }
    auto links_down = [&](int g) {
        auto it = passive.find(ids[(size_t)g]);
        return it != passive.end() && it->second.links_total > 0 && it->second.links_active < it->second.links_total;
    };
    int best = 0;
    for (int g = 1; g < G; ++g) {
        const int sb = row[(size_t)best] + col[(size_t)best], sg = row[(size_t)g] + col[(size_t)g];
        if (sg > sb || (sg == sb && links_down(g) && !links_down(best))) best = g;       // ties: links down first, then the lower position
    }
    if (row[(size_t)best] + col[(size_t)best] == 0) return out;
    out[key("nvlink-suspect")] = "gpu" + std::to_string(ids[(size_t)best]);
    const int r = row[(size_t)best], c = col[(size_t)best], half = (G - 1 + 1) / 2;
    if (links_down(best)) {
        const auto& st = passive.at(ids[(size_t)best]);
        const uint32_t mask = (uint32_t)(((1ull << st.links_total) - 1) & ~(uint64_t)st.active_mask);
        char hex[32];
        snprintf(hex, sizeof(hex), "0x%x", mask);
        out[key("nvlink-suspect-evidence")] = "links-down";
        out[key(ids[(size_t)best], "nvlink-links-down-mask")] = hex;
    } else if (G > 2 && r >= half && c >= half) out[key("nvlink-suspect-evidence")] = "port-both-directions";
    else if (G > 2 && r > c && r >= 2) out[key("nvlink-suspect-evidence")] = "egress-cold";
    else if (G > 2 && c > r && c >= 2) out[key("nvlink-suspect-evidence")] = "ingress-cold";
    else out[key("nvlink-suspect-evidence")] = "pair-only";
    return out;
}

inline std::string render(const Labels& l, double expiry_unix = 0) {
    std::string text;
    if (expiry_unix > 0) {               // NFD local source [RECALLED, NFD >= 0.14]: the labels of this file are dropped after this instant
        const time_t t = (time_t)expiry_unix;
        struct tm tmv;
        gmtime_r(&t, &tmv);
        char buf[64];
        strftime(buf, sizeof(buf), "%Y-%m-%dT%H:%M:%SZ", &tmv);
        text += std::string("# +expiry-time=") + buf + "\n";
    }
    for (const auto& kv : l) {                                         // std::map iterates sorted by key, like sorted(labels.items())
        if (!valid_label(kv.first, kv.second)) throw std::runtime_error("invalid label: " + kv.first + "=" + kv.second);
        text += kv.first + "=" + kv.second + "\n";
    }
    return text;
}

// Atomic replace (NFD may read at any time): write a hidden temp file, then rename.
inline void mkdirs(const std::string& dir) {
    for (size_t i = 1; i <= dir.size(); ++i)
        if (i == dir.size() || dir[i] == '/') ::mkdir(dir.substr(0, i).c_str(), 0755);
}

inline std::string write_feature_file(const Labels& l, const std::string& dir, const std::string& name = "b200probe", double expiry_unix = 0) {
    mkdirs(dir);
    const std::string text = render(l, expiry_unix);
    std::string tmpl = dir + "/.b200probe.XXXXXX";                       // dot-files are ignored by NFD
    std::vector<char> tmp(tmpl.begin(), tmpl.end());
    tmp.push_back(0);
    const int fd = ::mkstemp(tmp.data());
    if (fd < 0) throw std::runtime_error("mkstemp in " + dir + ": " + strerror(errno));
    bool ok = true;
    for (size_t off = 0; off < text.size() && ok;) {
        const ssize_t w = ::write(fd, text.data() + off, text.size() - off);
        if (w < 0) { if (errno == EINTR) continue; ok = false; }
        else off += (size_t)w;
    }
    ::fchmod(fd, 0644);
    ::close(fd);
    const std::string path = dir + "/" + name;
    if (!ok || ::rename(tmp.data(), path.c_str()) != 0) { ::unlink(tmp.data()); throw std::runtime_error("writing " + path + " failed"); }
    return path;
}

// This node's own healthy figures (first plausible healthy round), key=value lines under the state directory; twin of
// labels.py Calibration: accepted once, when within 15 % of the pool figure; the gate is then a fraction of THAT.
class Calibration {
public:
    explicit Calibration(const std::string& state_dir) : path_(state_dir + "/calibration"), dir_(state_dir) {
        std::ifstream f(path_);
        std::string line;
        while (std::getline(f, line)) {
            const size_t eq = line.find('=');
            if (line.empty() || line[0] == '#' || eq == std::string::npos) continue;
            char* end = nullptr;
            const double v = strtod(line.c_str() + eq + 1, &end);
            if (end && end != line.c_str() + eq + 1) vals_[line.substr(0, eq)] = v;
        }
    }
    double get(const std::string& k, double pool) const { auto it = vals_.find(k); return it == vals_.end() ? pool : it->second; }
    void offer(const std::string& k, double value, double pool) {
        if (vals_.count(k) || value < 0.85 * pool || value > 1.15 * pool) return;
        vals_[k] = value;
        mkdirs(dir_);
        const std::string tmp = path_ + ".tmp";
        { std::ofstream f(tmp); char buf[64]; for (const auto& kv : vals_) { snprintf(buf, sizeof(buf), "%.1f", kv.second); f << kv.first << "=" << buf << "\n"; } }
        ::rename(tmp.c_str(), path_.c_str());
    }
private:
    std::string path_, dir_;
    std::map<std::string, double> vals_;
};

// Runs the active probes on every enumerated, IDLE GPU at an interval and publishes the labels.  A probe that fails for a
// reason of the GPU (CUDA error, data mismatch, too slow) publishes ...healthy=false; a GPU that is in use or has no memory
// to spare is skipped and keeps its last idle verdict.  Never blocks ListAndWatch; holds no device memory between rounds.
class ActiveProbeRunner {
public:
    ActiveProbeRunner(const std::string& features_dir, double interval_s, bool run_nvlink = true, bool run_gemm = true, bool keep_arenas = false)
        : dir_(features_dir), interval_s_(interval_s), run_nvlink_(run_nvlink), run_gemm_(run_gemm), keep_arenas_(keep_arenas),
          cal_(getenv("B200PROBE_STATE_DIR") && *getenv("B200PROBE_STATE_DIR") ? std::string(getenv("B200PROBE_STATE_DIR")) : features_dir + "/.b200probe-state") {}
    ~ActiveProbeRunner() { stop(); }

    Labels run_once() {
        Labels l;
        int n = 0;
        b200probe_device_count(&n);
        std::vector<b200probe_device_t> infos((size_t)n);
        for (int i = 0; i < n; ++i) b200probe_device_info(i, &infos[(size_t)i]);
        // who is on the devices?  asked once, before any probe of ours shows up in the utilisation figures
        std::map<int, std::string> state;
        const char* ign = getenv("B200PROBE_IGNORE_TENANTS");            // benches / tests: the caller IS the tenant
        const bool ignore_tenants = ign && *ign && strcmp(ign, "0") != 0;
        for (const auto& d : infos) {
            b200probe_busy_t busy;
            state[d.index] = (!ignore_tenants && b200probe_device_busy(d.index, &busy) == 0 && busy.busy) ? "busy" : "probed";
        }
        const bool explicit_hbm = getenv("B200PROBE_HBM_MIN_GBS") != nullptr, explicit_gemm = getenv("B200PROBE_GEMM_MIN_TFLOPS") != nullptr;
        const bool explicit_gemm_fp8 = getenv("B200PROBE_GEMM_FP8_MIN_TFLOPS") != nullptr;

        for (const auto& d : infos) {
            if (state[d.index] != "probed") continue;
            b200probe_hbm_cfg_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.min_bytes = 1ull << 28; cfg.max_bytes = 1ull << 30; cfg.warmup = 2; cfg.reps = 5; cfg.verify = 1;
            std::vector<b200probe_hbm_result_t> pts(128);
            int got = 0;
            const int rc = b200probe_hbm_sweep(d.index, &cfg, pts.data(), (int)pts.size(), &got);
            if (rc == B200PROBE_ENOMEM) {
                state[d.index] = "no-memory";
                plugin::logf("GPU %d: no device memory for the HBM probe (tenants hold it): inconclusive", d.index);
            } else if (rc) {
                plugin::logf("HBM probe failed on GPU %d: %s", d.index, b200probe_strerror(rc));
                l[key(d.index, "hbm-healthy")] = "false";
            } else {
                pts.resize((size_t)got);
                Thresholds th = th_;
                const std::string ck = std::string("hbm-copy-gbs.") + d.uuid;
                if (!explicit_hbm) th.hbm_min_gbs = 0.90 * cal_.get(ck, kHbmMeasured);
                std::map<int, std::vector<b200probe_hbm_result_t>> one;
                one[d.index] = pts;
                Labels gl = hbm_labels(one, th);
                for (const auto& kv : gl) if (is_gpu_key(kv.first)) l[kv.first] = kv.second;
                auto h = gl.find(key(d.index, "hbm-healthy")), c = gl.find(key(d.index, "hbm-copy-gbs"));
                if (h != gl.end() && h->second == "true" && c != gl.end()) cal_.offer(ck, atof(c->second.c_str()), kHbmMeasured);
            }
        }
        if (run_gemm_) {
            for (const auto& d : infos) {
                if (state[d.index] != "probed") continue;
                b200probe_gemm_cfg_t cfg;
                memset(&cfg, 0, sizeof(cfg));
                cfg.warmup = 2; cfg.reps = 5;
                b200probe_gemm_result_t r;
                const int rc = b200probe_gemm(d.index, &cfg, &r);
                if (rc == B200PROBE_ENOMEM) state[d.index] = "no-memory";
                else if (rc) {
                    plugin::logf("GEMM probe failed on GPU %d: %s", d.index, b200probe_strerror(rc));
                    l[key(d.index, "gemm-healthy")] = "false";
                } else {
                    Thresholds th = th_;
                    const std::string ck = std::string("gemm-tflops.") + d.uuid;
                    if (!explicit_gemm) th.gemm_min_tflops = 0.70 * cal_.get(ck, kGemmMeasured);
                    std::map<int, b200probe_gemm_result_t> one;
                    one[d.index] = r;
                    Labels gl = gemm_labels(one, th);
                    for (const auto& kv : gl) if (is_gpu_key(kv.first)) l[kv.first] = kv.second;
                    auto h = gl.find(key(d.index, "gemm-healthy"));
                    if (h != gl.end() && h->second == "true") cal_.offer(ck, r.tflops_median, kGemmMeasured);
                }
            }
        }
        if (gemm_fp8_enabled()) {
            for (const auto& d : infos) {
                if (state[d.index] != "probed") continue;
                b200probe_gemm_cfg_t cfg;
                memset(&cfg, 0, sizeof(cfg));
                cfg.warmup = 2; cfg.reps = 5;
                b200probe_gemm_result_t r;
                const int rc = b200probe_gemm_fp8(d.index, &cfg, &r);
                if (rc == B200PROBE_ENOMEM) {
                    state[d.index] = "no-memory";
                    plugin::logf("GPU %d: no device memory for the FP8 GEMM probe (tenants hold it): inconclusive", d.index);
                } else if (rc) {
                    plugin::logf("FP8 GEMM probe failed on GPU %d: %s", d.index, b200probe_strerror(rc));
                    l[key(d.index, "gemm-fp8-healthy")] = "false";
                } else {
                    Thresholds th = th_;
                    const std::string ck = std::string("gemm-fp8-tflops.") + d.uuid;
                    if (!explicit_gemm_fp8) th.gemm_fp8_min_tflops = 0.70 * cal_.get(ck, kGemmFp8Measured);
                    std::map<int, b200probe_gemm_result_t> one;
                    one[d.index] = r;
                    Labels gl = gemm_fp8_labels(one, th);
                    for (const auto& kv : gl) if (is_gpu_key(kv.first)) l[kv.first] = kv.second;
                    auto h = gl.find(key(d.index, "gemm-fp8-healthy"));
                    if (h != gl.end() && h->second == "true") cal_.offer(ck, r.tflops_median, kGemmFp8Measured);
                }
            }
        }
        if (const double fraction = memtest_fraction(); fraction > 0) {
            for (const auto& d : infos) {
                if (state[d.index] != "probed") continue;
                b200probe_memtest_cfg_t cfg;
                memset(&cfg, 0, sizeof(cfg));
                cfg.fraction = fraction;
                b200probe_memtest_result_t r;
                const int rc = b200probe_hbm_memtest(d.index, &cfg, &r);
                if (rc == B200PROBE_ENOMEM) {
                    state[d.index] = "no-memory";
                    plugin::logf("GPU %d: no device memory for the HBM memtest (tenants hold it): inconclusive", d.index);
                } else if (rc) {
                    plugin::logf("HBM memtest failed on GPU %d: %s", d.index, b200probe_strerror(rc));
                    l[key(d.index, "hbm-memtest-healthy")] = "false";
                } else {
                    for (const auto& kv : memtest_labels(d.index, r)) l[kv.first] = kv.second;
                }
            }
        }
        // GPUs that were skipped keep what their last measured round said
        for (const auto& d : infos) {
            l[key(d.index, "probe-state")] = state[d.index];
            if (state[d.index] != "probed") { carry(&l, d.index, "hbm-"); carry(&l, d.index, "gemm-"); }
        }
        aggregate(&l, "hbm-healthy");
        aggregate(&l, "hbm-memtest-healthy");
        aggregate(&l, "gemm-fp8-healthy");
        if (run_gemm_) aggregate(&l, "gemm-healthy");
        {
            bool have = false;
            double mn = 0;
            for (const auto& kv : l) {
                int g; std::string leaf;
                if (split_gpu_key(kv.first, &g, &leaf) && leaf == "hbm-copy-gbs") { const double v = atof(kv.second.c_str()); mn = have ? std::min(mn, v) : v; have = true; }
            }
            if (have) l[key("hbm-copy-min-gbs")] = rint_str(mn);
        }

        // ---- NVLink: passive state of every GPU, the exchange over the idle ones ----
        std::map<int, b200probe_nvlink_status_t> before;
        for (const auto& d : infos) { b200probe_nvlink_status_t st; if (b200probe_nvlink_passive(d.index, &st) == 0) before[d.index] = st; }
        { Labels got = nvlink_passive_labels(before); for (const auto& kv : got) l[kv.first] = kv.second; }
        std::vector<int> ords, ids;
        for (int i = 0; i < n; ++i) {
            b200probe_device_t d;
            if (b200probe_device_info(i, &d) == 0 && d.cuda_ordinal >= 0 && state[d.index] == "probed") { ords.push_back(d.cuda_ordinal); ids.push_back(d.index); }
        }
        bool ran_nvlink = false;
        if (run_nvlink_ && ords.size() >= 2) {
            const int G = (int)ords.size();
            b200probe_a2a_cfg_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.warmup = 2; cfg.reps = 5; cfg.verify = 1;
            std::vector<double> pair((size_t)(G * G), 0.0);
            b200probe_a2a_result_t rep;
            const int rc = b200probe_nvlink_a2a(ords.data(), G, &cfg, pair.data(), &rep);
            if (rc == B200PROBE_ENOMEM) {
                plugin::logf("no device memory for the NVLink exchange: inconclusive");
            } else if (rc) {
                plugin::logf("NVLink probe failed: %s", b200probe_strerror(rc));
                l[key("nvlink-healthy")] = "false";
                ran_nvlink = true;
            } else {
                ran_nvlink = true;
                Labels got = nvlink_labels(rep, pair, th_, ids);
                for (const auto& kv : got) l[kv.first] = kv.second;
                got = nvlink_localise(rep, pair, ids, before);
                for (const auto& kv : got) l[kv.first] = kv.second;
                auto it = l.find(key("nvlink-links-ok"));
                if (it != l.end() && it->second == "false") l[key("nvlink-healthy")] = "false";   // a dead link fails the gate even if the matrix clears the bar
                double min_eff = 2.0;
                for (int idx : ids) {
                    auto bi = before.find(idx);
                    b200probe_nvlink_status_t after;
                    if (bi == before.end() || b200probe_nvlink_passive(idx, &after) != 0 || !bi->second.counters_ok || !after.counters_ok) continue;
                    const double dd = (double)(after.data_tx_kib - bi->second.data_tx_kib), rr = (double)(after.raw_tx_kib - bi->second.raw_tx_kib);
                    if (rr > 0 && dd > 0) min_eff = std::min(min_eff, dd / rr);
                }
                if (min_eff <= 1.0) l[key("nvlink-data-over-raw-pct")] = rint_str(100.0 * min_eff);
            }
        }
        if (run_nvlink_ && !ran_nvlink) {
            // nothing measured this round (GPUs busy / a single GPU): the whole NVLink picture of the last measured round stands
            for (const auto& kv : last_)
                if (kv.first.find("nvlink-") != std::string::npos && kv.first.find("nvlink-links-") == std::string::npos && !l.count(kv.first)) l[kv.first] = kv.second;
        }
        gate_label(&l);
        if (!keep_arenas_) release(infos);
        last_ = l;
        write_feature_file(l, dir_, "b200probe", (double)time(nullptr) + 2.0 * interval_s_ + 60.0);
        return l;
    }

    // free every probe arena of this process (device memory, streams, NCCL communicators)
    static void release(const std::vector<b200probe_device_t>& infos) {
        for (const auto& d : infos) if (d.cuda_ordinal >= 0) { b200probe_hbm_release(d.cuda_ordinal); b200probe_gemm_release(d.cuda_ordinal); }
        b200probe_a2a_release();
    }

    // clean shutdown: the verdicts are no longer maintained, so they are removed (NFD drops the labels)
    void withdraw() { ::unlink((dir_ + "/b200probe").c_str()); }

    void start() {
        stop_ = false;
        started_ = true;
        thread_ = std::thread([this] {
            while (!stop_) {
                try { run_once(); } catch (const std::exception& e) { plugin::logf("active probe round failed: %s", e.what()); }
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait_for(lk, std::chrono::milliseconds((long long)(interval_s_ * 1000)), [this] { return stop_.load(); });
            }
        });
    }
    void stop() {
        { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }      // under the mutex: the loop cannot test the predicate and then miss the notify
        cv_.notify_all();
        if (thread_.joinable()) thread_.join();
        if (started_) { withdraw(); started_ = false; }
    }

private:
    static bool split_gpu_key(const std::string& k, int* gpu, std::string* leaf) {
        const std::string pfx = std::string(kPrefix) + "gpu";
        if (k.compare(0, pfx.size(), pfx) != 0) return false;
        size_t i = pfx.size();
        if (i >= k.size() || !isdigit((unsigned char)k[i])) return false;
        int g = 0;
        while (i < k.size() && isdigit((unsigned char)k[i])) g = g * 10 + (k[i++] - '0');
        if (i >= k.size() || k[i] != '.') return false;
        *gpu = g; *leaf = k.substr(i + 1);
        return true;
    }
    static bool is_gpu_key(const std::string& k) { int g; std::string leaf; return split_gpu_key(k, &g, &leaf); }
    void carry(Labels* l, int idx, const char* leaf_prefix) const {
        for (const auto& kv : last_) {
            int g; std::string leaf;
            if (split_gpu_key(kv.first, &g, &leaf) && g == idx && leaf.compare(0, strlen(leaf_prefix), leaf_prefix) == 0 && !l->count(kv.first)) (*l)[kv.first] = kv.second;
        }
    }
    static void aggregate(Labels* l, const char* leaf_name) {
        bool any = false, all = true;
        for (const auto& kv : *l) {
            int g; std::string leaf;
            if (split_gpu_key(kv.first, &g, &leaf) && leaf == leaf_name) { any = true; all = all && kv.second == "true"; }
        }
        if (any) (*l)[key(leaf_name)] = b(all); else l->erase(key(leaf_name));
    }

    std::string dir_;
    double interval_s_;
    bool run_nvlink_, run_gemm_, keep_arenas_;
    Calibration cal_;
    Thresholds th_;
    Labels last_;
    bool started_ = false;
    std::atomic<bool> stop_{false};
    std::mutex mu_;
    std::condition_variable cv_;
    std::thread thread_;
};

}  // namespace labels
