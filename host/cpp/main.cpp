// b200-device-plugin — the container entry point that stands where the upstream plugin binary stands inside
// the nvdp DaemonSet (/root/reference/README.md:116): reads the plugin config document the chart mounts
// (/root/reference/values.yaml:8-18), serves the kubelet device-plugin API v1beta1 on a unix socket,
// registers with kubelet, follows the passive XID/ECC health events, and (unless --no-active-probe) runs the
// B200 active probes at an interval and publishes their verdicts as NFD labels.
//
//   b200-device-plugin --config-file /config/config.yaml
//   b200-device-plugin --check-config FILE          print the parsed configuration as JSON (parity tests)
//   b200-device-plugin --check-values FILE          the same for the chart's values.yaml (gfd, runtimeClassName, config.map)
//   b200-device-plugin --probe-once                 one active-probe round, labels on stdout
//   b200-device-plugin --probe-rounds N             N rounds of one runner, labels after each (tests)
#include <signal.h>

#include <fstream>
#include <iostream>
#include <sstream>

#include "labels.hpp"
#include "plugin.hpp"

static std::atomic<bool> g_stop{false}, g_reload{false};
static void on_signal(int sig) { if (sig == SIGHUP) g_reload = true; else g_stop = true; }

static std::string json_str(const std::string& s) {
    std::string o = "\"";
    for (unsigned char c : s) {
        if (c == '"' || c == '\\') { o += '\\'; o += (char)c; }
        else if (c < 0x20 || c >= 0x7f) { char b[8]; snprintf(b, sizeof(b), "\\u%04x", c); o += b; }
        else o += (char)c;
    }
    return o + "\"";
}

// stdin: one hex-encoded header block per line, decoded by ONE decoder in order (dynamic-table continuity);
// stdout: one JSON array of [name, value] pairs per block, or {"error": ...}.  Transport self-check used by the tests.
static int hpack_decode_stdin() {
    hpack::Decoder dec;
    std::string line;
    while (std::getline(std::cin, line)) {
        std::string bytes;
        for (size_t i = 0; i + 1 < line.size(); i += 2) bytes.push_back((char)strtol(line.substr(i, 2).c_str(), nullptr, 16));
        std::vector<hpack::Header> hs;
        if (!dec.decode((const uint8_t*)bytes.data(), bytes.size(), &hs)) { printf("{\"error\":\"decode failed\"}\n"); continue; }
        std::string o = "[";
        for (size_t i = 0; i < hs.size(); ++i) o += std::string(i ? "," : "") + "[" + json_str(hs[i].first) + "," + json_str(hs[i].second) + "]";
        printf("%s]\n", o.c_str());
    }
    return 0;
}

// --labels-from-stdin: synthetic probe results in, rendered feature file out (CPU parity check of labels.hpp against
// labels.py).  One record per line:
//   hbm <gpu> <bytes> <mode 1|2|4> <gbs_median> <verified> <cache_resident>
//   gemm <gpu> <tflops_median> <verified>
//   passive <gpu> <links_total> <links_active> <fabric_state> <fabric_status> <fabric_health_mask> [<active_mask>]
//   a2a <G> <verified> <min_pair_gbs> <G egress> <G ingress> <G*G pair, row-major>
//   a2ax <pair_source> <G ids>        (optional, after a2a: what the matrix holds and the NVML index of every position -> nvlink_localise)
//   gemm_fp8 <gpu> <tflops_median> <verified>
//   memtest <gpu> <bytes_tested> <bad_words> <ecc_corrected_delta> <ecc_uncorrected_delta> <remap_pending> <remap_failure>
static int labels_from_stdin() {
    std::map<int, std::vector<b200probe_hbm_result_t>> hbm;
    std::map<int, b200probe_gemm_result_t> gemm, gemm_fp8;
    std::map<int, b200probe_nvlink_status_t> passive;
    std::map<int, b200probe_memtest_result_t> memtest;
    bool have_a2a = false;
    b200probe_a2a_result_t rep;
    std::vector<double> pair;
    std::vector<int> ids;
    memset(&rep, 0, sizeof(rep));
    std::string line;
    while (std::getline(std::cin, line)) {
        std::istringstream in(line);
        std::string kind;
        in >> kind;
        if (kind == "hbm") {
            int gpu; b200probe_hbm_result_t r;
            memset(&r, 0, sizeof(r));
            unsigned long long bytes;
            in >> gpu >> bytes >> r.mode >> r.gbs_median >> r.verified >> r.cache_resident;
            r.bytes = bytes;
            hbm[gpu].push_back(r);
        } else if (kind == "gemm") {
            int gpu; b200probe_gemm_result_t r;
            memset(&r, 0, sizeof(r));
            in >> gpu >> r.tflops_median >> r.verified;
            gemm[gpu] = r;
        } else if (kind == "gemm_fp8") {
            int gpu; b200probe_gemm_result_t r;
            memset(&r, 0, sizeof(r));
            in >> gpu >> r.tflops_median >> r.verified;
            gemm_fp8[gpu] = r;
        } else if (kind == "passive") {
            int gpu; b200probe_nvlink_status_t st;
            memset(&st, 0, sizeof(st));
            in >> gpu >> st.links_total >> st.links_active >> st.fabric_state >> st.fabric_status >> st.fabric_health_mask;
            unsigned mask = 0;
            if (in >> mask) st.active_mask = mask;
            passive[gpu] = st;
        } else if (kind == "a2a") {
            in >> rep.g >> rep.verified >> rep.min_pair_gbs;
            for (int i = 0; i < rep.g; ++i) in >> rep.egress_gbs[i];
            for (int i = 0; i < rep.g; ++i) in >> rep.ingress_gbs[i];
            pair.assign((size_t)(rep.g * rep.g), 0.0);
            for (auto& v : pair) in >> v;
            have_a2a = true;
        } else if (kind == "memtest") {
            int gpu; b200probe_memtest_result_t r;
            memset(&r, 0, sizeof(r));
            unsigned long long bytes, bad;
            long long corr, unc;
            in >> gpu >> bytes >> bad >> corr >> unc >> r.ecc_after.remap_pending >> r.ecc_after.remap_failure;
            r.bytes_tested = bytes; r.bad_words = bad; r.ecc_corrected_delta = corr; r.ecc_uncorrected_delta = unc;
            memtest[gpu] = r;
        } else if (kind == "a2ax") {
            in >> rep.pair_source;
            ids.assign((size_t)rep.g, 0);
            for (auto& v : ids) in >> v;
        }
    }
    labels::Thresholds th;
    labels::Labels l;
    auto merge = [&](const labels::Labels& got) { for (const auto& kv : got) l[kv.first] = kv.second; };
    if (!hbm.empty()) merge(labels::hbm_labels(hbm, th));
    if (!gemm.empty()) merge(labels::gemm_labels(gemm, th));
    if (!gemm_fp8.empty()) merge(labels::gemm_fp8_labels(gemm_fp8, th));
    merge(labels::nvlink_passive_labels(passive));
    for (const auto& kv : memtest) merge(labels::memtest_labels(kv.first, kv.second));
    if (!memtest.empty()) {
        bool all = true;
        for (const auto& kv : l) if (kv.first.size() > 20 && kv.first.compare(kv.first.size() - 20, 20, ".hbm-memtest-healthy") == 0) all = all && kv.second == "true";
        l[labels::key("hbm-memtest-healthy")] = labels::b(all);
    }
    if (have_a2a) {
        merge(labels::nvlink_labels(rep, pair, th, ids));
        if (!ids.empty()) merge(labels::nvlink_localise(rep, pair, ids, passive));
    }
    labels::gate_label(&l);
    fputs(labels::render(l).c_str(), stdout);
    return 0;
}

static std::string config_json(const config::PluginConfig& c);

// --check-values FILE: the Helm values file of the reference, parsed like config.py's parse_helm_values
static int check_values(const std::string& path) {
    std::ifstream f(path);
    std::stringstream ss;
    ss << f.rdbuf();
    try {
        const config::HelmValues v = config::parse_helm_values(ss.str());
        std::string cfgs = "{", raws = "{";
        for (size_t i = 0; i < v.configs.size(); ++i) {
            cfgs += std::string(i ? "," : "") + json_str(v.configs[i].first) + ":" + config_json(v.configs[i].second);
            raws += std::string(i ? "," : "") + json_str(v.raw_configs[i].first) + ":" + json_str(v.raw_configs[i].second);
        }
        printf("{\"ok\":true,\"gfd_enabled\":%s,\"runtime_class_name\":%s,\"configs\":%s},\"raw_configs\":%s},\"default\":%s}\n", v.gfd_enabled ? "true" : "false",
               v.runtime_class_name.empty() ? "null" : json_str(v.runtime_class_name).c_str(), cfgs.c_str(), raws.c_str(), config_json(v.default_config()).c_str());
    } catch (const config::Error& e) {
        printf("{\"ok\":false,\"error\":%s}\n", json_str(e.what()).c_str());
    }
    return 0;
}

static std::string config_json(const config::PluginConfig& c) {
    std::string res = "[";
    for (size_t i = 0; i < c.time_slicing.resources.size(); ++i) {
        const auto& r = c.time_slicing.resources[i];
        res += std::string(i ? "," : "") + "{\"name\":" + json_str(r.name) + ",\"replicas\":" + std::to_string(r.replicas) +
               ",\"rename\":" + (r.rename.empty() ? "null" : json_str(r.rename)) + "}";
    }
    res += "]";
    return "{\"version\":" + json_str(c.version) + ",\"mig_strategy\":" + json_str(c.mig_strategy) + ",\"rename_by_default\":" +
           (c.time_slicing.rename_by_default ? "true" : "false") + ",\"fail_requests_greater_than_one\":" +
           (c.time_slicing.fail_requests_greater_than_one ? "true" : "false") + ",\"resources\":" + res + ",\"resource_name\":" + json_str(c.resource_name()) +
           ",\"replicas\":" + std::to_string(c.replicas()) + ",\"is_shared\":" + (c.is_shared() ? "true" : "false") + "}";
}

static int check_config(const std::string& path) {
    std::ifstream f(path);
    std::stringstream ss;
    ss << f.rdbuf();
    try {
        const config::PluginConfig c = config::parse_plugin_config(ss.str());
        std::string res = "[";
        for (size_t i = 0; i < c.time_slicing.resources.size(); ++i) {
            const auto& r = c.time_slicing.resources[i];
            res += std::string(i ? "," : "") + "{\"name\":" + json_str(r.name) + ",\"replicas\":" + std::to_string(r.replicas) +
                   ",\"rename\":" + (r.rename.empty() ? "null" : json_str(r.rename)) + "}";
        }
        res += "]";
        printf("{\"ok\":true,\"version\":%s,\"mig_strategy\":%s,\"device_list_strategy\":%s,\"device_id_strategy\":%s,\"pass_device_specs\":%s,"
               "\"rename_by_default\":%s,\"fail_requests_greater_than_one\":%s,\"resources\":%s,\"resource_name\":%s,\"replicas\":%lld,\"is_shared\":%s}\n",
               json_str(c.version).c_str(), json_str(c.mig_strategy).c_str(), json_str(c.device_list_strategy).c_str(), json_str(c.device_id_strategy).c_str(),
               c.pass_device_specs ? "true" : "false", c.time_slicing.rename_by_default ? "true" : "false",
               c.time_slicing.fail_requests_greater_than_one ? "true" : "false", res.c_str(), json_str(c.resource_name()).c_str(), (long long)c.replicas(),
               c.is_shared() ? "true" : "false");
        return 0;
    } catch (const config::Error& e) {
        printf("{\"ok\":false,\"error\":%s}\n", json_str(e.what()).c_str());
        return 0;
    }
}

int main(int argc, char** argv) {
    std::string config_file = getenv("CONFIG_FILE") ? getenv("CONFIG_FILE") : "/config/config.yaml";
    std::string socket_dir = v1beta1::kDevicePluginPath, kubelet_socket, nvml_path;
    std::string features_dir = "/etc/kubernetes/node-feature-discovery/features.d";
    double probe_interval = getenv("B200PROBE_INTERVAL_S") ? atof(getenv("B200PROBE_INTERVAL_S")) : 600.0, watch_period = 1.0;
    bool active = true, probe_once = false, health = true;
    int probe_rounds = 1;
    int health_timeout_ms = 5000;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&](std::string* out) { if (i + 1 >= argc) { fprintf(stderr, "%s needs a value\n", a.c_str()); exit(2); } *out = argv[++i]; };
        std::string v;
        if (a == "--check-config") { val(&v); return check_config(v); }
        else if (a == "--check-values") { val(&v); return check_values(v); }
        else if (a == "--labels-from-stdin") return labels_from_stdin();
        else if (a == "--hpack-decode") return hpack_decode_stdin();
        else if (a == "--config-file") val(&config_file);
        else if (a == "--socket-dir") val(&socket_dir);
        else if (a == "--kubelet-socket") val(&kubelet_socket);
        else if (a == "--features-dir") val(&features_dir);
        else if (a == "--nvml-path") val(&nvml_path);
        else if (a == "--probe-interval") { val(&v); probe_interval = atof(v.c_str()); }
        else if (a == "--watch-period") { val(&v); watch_period = atof(v.c_str()); }
        else if (a == "--health-timeout-ms") { val(&v); health_timeout_ms = atoi(v.c_str()); }
        else if (a == "--no-active-probe") active = false;
        else if (a == "--no-health") health = false;
        else if (a == "--probe-once") probe_once = true;
        else if (a == "--probe-rounds") { val(&v); probe_once = true; probe_rounds = std::max(1, atoi(v.c_str())); }   // N rounds of ONE runner (tests: carry-over, calibration)
        else if (a == "--version") { printf("b200-device-plugin abi %d\n", b200probe_abi_version()); return 0; }
        else { fprintf(stderr, "unknown argument %s\n", a.c_str()); return 2; }
    }
    int rc = b200probe_init(nvml_path.empty() ? nullptr : nvml_path.c_str());
    if (rc) { plugin::logf("b200probe_init failed: %s", b200probe_strerror(rc)); return 1; }
    if (probe_once) {
        try {
            labels::ActiveProbeRunner runner(features_dir, 0);
            for (int r = 0; r < probe_rounds; ++r) {
                if (probe_rounds > 1) printf("== round %d\n", r);
                fputs(labels::render(runner.run_once()).c_str(), stdout);
            }
            return 0;
        } catch (const std::exception& e) { plugin::logf("probe round failed: %s", e.what()); return 1; }
    }
    config::PluginConfig cfg;
    try {
        std::ifstream f(config_file);
        if (!f) throw config::Error("cannot open " + config_file);
        std::stringstream ss;
        ss << f.rdbuf();
        cfg = config::parse_plugin_config(ss.str());
    } catch (const std::exception& e) { plugin::logf("config: %s", e.what()); return 1; }

    struct sigaction sa;
    memset(&sa, 0, sizeof(sa));
    sa.sa_handler = on_signal;
    sigaction(SIGTERM, &sa, nullptr);
    sigaction(SIGINT, &sa, nullptr);
    signal(SIGPIPE, SIG_IGN);
    sigaction(SIGHUP, &sa, nullptr);
    try {
        std::unique_ptr<plugin::DevicePlugin> dp(new plugin::DevicePlugin(cfg, socket_dir, kubelet_socket, health_timeout_ms));
        dp->start(watch_period, health);
        std::unique_ptr<labels::ActiveProbeRunner> runner;
        if (active) { runner.reset(new labels::ActiveProbeRunner(features_dir, probe_interval)); runner->start(); }
        plugin::logf("serving '%s' on %s (%zu devices)", dp->resource().c_str(), dp->socket_path().c_str(), dp->devices().size());
        while (!g_stop) {
            usleep(100000);
            if (!g_reload.exchange(false)) continue;
            // SIGHUP: the chart's config-manager sidecar rewrote the config file [RECALLED]; take the new document if it
            // parses (a bad one keeps the running configuration), re-enumerate, serve again and re-Register.
            try {
                std::ifstream f(config_file);
                if (!f) throw config::Error("cannot open " + config_file);
                std::stringstream ss;
                ss << f.rdbuf();
                const config::PluginConfig fresh = config::parse_plugin_config(ss.str());
                dp->stop();
                dp.reset();
                b200probe_health_close();
                dp.reset(new plugin::DevicePlugin(fresh, socket_dir, kubelet_socket, health_timeout_ms));
                dp->start(watch_period, health);
                plugin::logf("reloaded %s: serving '%s' on %s (%zu devices)", config_file.c_str(), dp->resource().c_str(), dp->socket_path().c_str(),
                             dp->devices().size());
            } catch (const config::Error& e) {
                plugin::logf("reload of %s rejected, keeping the running configuration: %s", config_file.c_str(), e.what());
            }
        }
        if (runner) runner->stop();
        if (dp) dp->stop();
    } catch (const std::exception& e) { plugin::logf("fatal: %s", e.what()); b200probe_shutdown(); return 1; }
    b200probe_shutdown();
    return 0;
}
