#include "conf.h"

#include <math.h>
#include <stdlib.h>
#include <unistd.h>

#include <fstream>
#include <sstream>

namespace cv {

static std::string trim(const std::string& s) {
    size_t a = 0, b = s.size();
    while (a < b && isspace(static_cast<unsigned char>(s[a]))) a++;
    while (b > a && isspace(static_cast<unsigned char>(s[b - 1]))) b--;
    return s.substr(a, b - a);
}

// ByteUnit::from_str (orpc/src/common/byte_unit.rs:76-125): binary units, case-insensitive
Err parse_byte_size(const std::string& in, int64_t* out) {
    std::string s = trim(in);
    for (auto& c : s) c = static_cast<char>(toupper(static_cast<unsigned char>(c)));
    if (s.empty()) return Err::common(" is not a valid size.");
    size_t n = 0;
    while (n < s.size() && (isdigit(static_cast<unsigned char>(s[n])) || s[n] == '.' || s[n] == 'E' || s[n] == '-' || s[n] == '+')) n++;
    // "E" is ambiguous with the EB unit only in theory; the reference list stops at PB
    std::string num = s.substr(0, n), unit = trim(s.substr(n));
    uint64_t mul;
    if (unit == "K" || unit == "KB") mul = 1ull << 10;
    else if (unit == "M" || unit == "MB") mul = 1ull << 20;
    else if (unit == "G" || unit == "GB") mul = 1ull << 30;
    else if (unit == "T" || unit == "TB") mul = 1ull << 40;
    else if (unit == "P" || unit == "PB") mul = 1ull << 50;
    else if (unit == "B" || unit.empty()) mul = 1;
    else return Err::common("only B, KB,, MB, GB, TB, PB are supported: " + s);
    if (num.empty()) return Err::common("invalid size string: " + s);
    char* end = nullptr;
    const double v = strtod(num.c_str(), &end);
    if (end == num.c_str() || *end) return Err::common("invalid size string: " + s);
    *out = static_cast<int64_t>(llround(v * static_cast<double>(mul)));
    return Err::ok();
}

Err ClientConf::init() {
    if (read_slice_size <= 0) read_slice_size = read_chunk_num * read_chunk_size;
    if (read_ahead_len <= 0) read_ahead_len = read_chunk_num * read_chunk_size;
    if (read_chunk_num <= 1 || read_ahead_len < 256 * 1024) enable_read_ahead = false;
    if (hostname.empty()) {
        if (const char* h = getenv("CURVINE_CLIENT_HOSTNAME")) hostname = h;
        else {
            char buf[256] = {0};
            gethostname(buf, sizeof(buf) - 1);
            hostname = buf;
        }
    }
    return Err::ok();
}

static std::string unquote(const std::string& v) {
    if (v.size() >= 2 && ((v.front() == '"' && v.back() == '"') || (v.front() == '\'' && v.back() == '\''))) return v.substr(1, v.size() - 2);
    return v;
}

Err parse_duration_ms(const std::string& in, int64_t* out) {
    std::string s;
    for (char c : in) s += static_cast<char>(tolower(static_cast<unsigned char>(c)));
    size_t a = 0, b = s.size();
    while (a < b && isspace(static_cast<unsigned char>(s[a]))) a++;
    while (b > a && isspace(static_cast<unsigned char>(s[b - 1]))) b--;
    s = s.substr(a, b - a);
    size_t k = 0;
    while (k < s.size() && (isdigit(static_cast<unsigned char>(s[k])) || s[k] == '.' || s[k] == 'e' || s[k] == '-' || s[k] == '+')) k++;
    const std::string num = s.substr(0, k);
    std::string unit = s.substr(k);
    while (!unit.empty() && isspace(static_cast<unsigned char>(unit.front()))) unit.erase(unit.begin());
    double mult;
    if (unit == "s" || unit == "second") mult = 1000.0;
    else if (unit == "m" || unit == "minute") mult = 60.0 * 1000;
    else if (unit == "h" || unit == "hour") mult = 3600.0 * 1000;
    else if (unit == "d" || unit == "day") mult = 86400.0 * 1000;
    else if (unit == "ms" || unit.empty()) mult = 1.0;
    else return Err::common("valid duration " + s + ", only d, h, m, s, ms are supported");
    if (num.empty()) return Err::common("invalid duration string: " + s);
    char* end = nullptr;
    const double v = strtod(num.c_str(), &end);
    if (end == num.c_str() || *end != '\0' || v < 0) return Err::common("invalid duration string: " + s);
    *out = static_cast<int64_t>(v * mult);
    return Err::ok();
}

static Err as_size(const std::string& v, int64_t* out) { return parse_byte_size(unquote(v), out); }
static bool as_bool(const std::string& v) { return unquote(v) == "true" || unquote(v) == "1"; }
static int64_t as_int(const std::string& v) { return strtoll(unquote(v).c_str(), nullptr, 10); }

static std::vector<std::string> as_list(const std::string& v) {
    std::vector<std::string> out;
    std::string s = trim(v);
    if (!s.empty() && s.front() == '[' && s.back() == ']') s = s.substr(1, s.size() - 2);
    else {
        out.push_back(unquote(s));
        return out;
    }
    // split on commas outside quotes
    std::string cur;
    bool inq = false;
    for (char c : s) {
        if (c == '"') inq = !inq;
        if (c == ',' && !inq) {
            if (!trim(cur).empty()) out.push_back(unquote(trim(cur)));
            cur.clear();
        } else cur.push_back(c);
    }
    if (!trim(cur).empty()) out.push_back(unquote(trim(cur)));
    return out;
}

// A deliberately small TOML subset: [section] headers, key = value, # comments, one-line arrays.
Err ClusterConf::from_string(const std::string& toml, ClusterConf* c) {
    std::istringstream in(toml);
    std::string line, section;
    while (std::getline(in, line)) {
        bool inq = false;
        for (size_t i = 0; i < line.size(); i++) {
            if (line[i] == '"') inq = !inq;
            if (line[i] == '#' && !inq) {
                line.resize(i);
                break;
            }
        }
        line = trim(line);
        if (line.empty()) continue;
        if (line.front() == '[' && line.find('=') == std::string::npos) {
            section = trim(line.substr(1, line.size() - 2));
            continue;
        }
        const size_t eq = line.find('=');
        if (eq == std::string::npos) return Err::common("bad conf line: " + line);
        const std::string k = trim(line.substr(0, eq)), v = trim(line.substr(eq + 1));
        Err e;
        if (section.empty()) {
            if (k == "cluster_id") c->cluster_id = unquote(v);
            else if (k == "namespace_manifest") c->namespace_manifest = unquote(v);
        } else if (section == "client") {
            ClientConf& cl = c->client;
            if (k == "block_size") e = as_size(v, &cl.block_size);
            else if (k == "read_chunk_size") e = as_size(v, &cl.read_chunk_size);
            else if (k == "read_chunk_num") cl.read_chunk_num = as_int(v);
            else if (k == "read_parallel") cl.read_parallel = as_int(v);
            else if (k == "read_slice_size") e = as_size(v, &cl.read_slice_size);
            else if (k == "short_circuit") cl.short_circuit = as_bool(v);
            else if (k == "enable_read_ahead") cl.enable_read_ahead = as_bool(v);
            else if (k == "read_ahead_len") e = as_size(v, &cl.read_ahead_len);
            else if (k == "drop_cache_len") e = as_size(v, &cl.drop_cache_len);
            else if (k == "max_cache_block_handles") cl.max_cache_block_handles = as_int(v);
            else if (k == "enable_smart_prefetch") cl.enable_smart_prefetch = as_bool(v);
            else if (k == "large_file_size") e = as_size(v, &cl.large_file_size);
            else if (k == "max_read_parallel") cl.max_read_parallel = as_int(v);
            else if (k == "sequential_read_threshold") cl.sequential_read_threshold = as_int(v);
            else if (k == "conn_timeout_ms") cl.conn_timeout_ms = as_int(v);
            else if (k == "rpc_timeout_ms") cl.rpc_timeout_ms = as_int(v);
            else if (k == "data_timeout_ms") cl.data_timeout_ms = as_int(v);
            else if (k == "enable_block_conn_pool") cl.enable_block_conn_pool = as_bool(v);
            else if (k == "block_conn_idle_size") cl.block_conn_idle_size = as_int(v);
            else if (k == "block_conn_idle_time") e = parse_duration_ms(unquote(v), &cl.block_conn_idle_time_ms);
            else if (k == "failed_worker_ttl") e = parse_duration_ms(unquote(v), &cl.failed_worker_ttl_ms);
            else if (k == "hostname") cl.hostname = unquote(v);
        } else if (section == "worker") {
            if (k == "data_dir") c->worker_dirs = as_list(v);
            else if (k == "hostname") c->worker_hostname = unquote(v);
            else if (k == "rpc_port") c->worker_port = static_cast<int>(as_int(v));
            else if (k == "enable_send_file") c->worker_enable_send_file = as_bool(v);
            else if (k == "mem_arena") c->worker_mem_arena = as_bool(v);
            else if (k == "arena_segment") e = as_size(v, &c->worker_arena_segment);
            else if (k == "arena_numa") {
                c->worker_arena_numa.clear();
                for (const auto& x : as_list(v)) c->worker_arena_numa.push_back(static_cast<int>(as_int(x)));
            } else if (k == "arena_reuse_delay") e = parse_duration_ms(unquote(v), &c->worker_arena_reuse_delay_ms);
            else if (k == "hbm_capacity") e = as_size(v, &c->worker_hbm_capacity);
            else if (k == "hbm_promote_after") c->worker_hbm_promote_after = static_cast<int>(as_int(v));
            else if (k == "hbm_device") c->worker_hbm_device = static_cast<int>(as_int(v));
        } else if (section == "b200") {
            B200Conf& b = c->b200;
            if (k == "device") b.device = static_cast<int>(as_int(v));
            else if (k == "fetch_threads") b.fetch_threads = static_cast<int>(as_int(v));
            else if (k == "pinned_slots") b.pinned_slots = static_cast<int>(as_int(v));
            else if (k == "verify_poly") b.verify_poly = static_cast<int>(as_int(v));
            else if (k == "verify") b.verify = as_bool(v);
            else if (k == "verify_batch") b.verify_batch = static_cast<int>(as_int(v));
            else if (k == "copy_streams") b.copy_streams = static_cast<int>(as_int(v));
            else if (k == "copy_group") b.copy_group = static_cast<int>(as_int(v));
            else if (k == "gpu_chunk_size") e = as_size(v, &b.gpu_chunk_size);
            else if (k == "numa_node") b.numa_node = static_cast<int>(as_int(v));
            else if (k == "zero_copy") b.zero_copy = as_bool(v);
            else if (k == "register_cache") e = as_size(v, &b.register_cache);
            else if (k == "register_min_age") e = parse_duration_ms(unquote(v), &b.register_min_age_ms);
            else if (k == "register_threads") b.register_threads = static_cast<int>(as_int(v));
            else if (k == "register_when_idle") b.register_when_idle = as_bool(v);
            else if (k == "gds") {
                const std::string m = unquote(v);
                if (m == "off" || m == "false" || m == "0") b.gds = false;
                else if (m == "auto") b.gds = true;
                else if (m == "on" || m == "true" || m == "1")
                    e = Err::common("gds = \"" + m + "\" (cuFile's compatibility mode) is not supported: use \"auto\" (GPUDirect Storage where nvidia-fs is loaded) or \"off\"");
                else e = Err::common("gds must be \"off\" or \"auto\": " + m);
            } else if (k == "local_unix_socket") b.local_unix_socket = as_bool(v);
            else if (k == "socket_buffer") e = as_size(v, &b.socket_buffer);
            else if (k == "arena") b.arena = as_bool(v);
            else if (k == "arena_preregister") b.arena_dirs = as_list(v);
            else if (k == "arena_register_slice") e = as_size(v, &b.arena_register_slice);
        }
        if (e) return e.ctx("conf key " + k);
    }
    return c->client.init();
}

Err ClusterConf::from_file(const std::string& path, ClusterConf* out) {
    std::ifstream f(path);
    if (!f) return Err(kFileNotFound, "conf file not found: " + path);
    std::stringstream ss;
    ss << f.rdbuf();
    CV_RETURN_IF_ERR(from_string(ss.str(), out));
    // environment beats the file, as in ClusterConf::from (curvine-common/src/conf/cluster_conf.rs:82-94)
    if (const char* h = getenv("CURVINE_WORKER_HOSTNAME")) out->worker_hostname = h;
    if (const char* h = getenv("CURVINE_CLIENT_HOSTNAME")) out->client.hostname = h;
    return Err::ok();
}

}  // namespace cv
