// Client/worker configuration: the reference's read knobs with the reference's defaults, plus the
// [b200] section this implementation adds.
//
// Mirrors curvine-common/src/conf/client_conf.rs:228-281,315-420 (defaults + init()),
// orpc/src/common/byte_unit.rs:29-34 (binary size strings: KB = 2^10 ...),
// curvine-common/src/conf/worker_conf.rs:59-95,176-207 (data_dir tags "[MEM:10MB]/path", enable_send_file).
#pragma once
#include <map>
#include <vector>

#include "common.h"

namespace cv {

struct ClientConf {
    int64_t block_size = 128ll << 20;
    int64_t read_chunk_size = 128 << 10;
    int64_t read_chunk_num = 8;
    int64_t read_parallel = 1;
    int64_t read_slice_size = 0;  // 0 -> chunk_num * chunk_size
    bool short_circuit = true;
    bool enable_read_ahead = true;
    int64_t read_ahead_len = 0;  // 0 -> chunk_num * chunk_size
    int64_t drop_cache_len = 1 << 20;
    int64_t max_cache_block_handles = 10;
    bool enable_smart_prefetch = true;
    int64_t large_file_size = 10ll << 30;
    int64_t max_read_parallel = 8;
    int64_t sequential_read_threshold = 7;
    int64_t conn_timeout_ms = 30 * 1000;   // client_conf.rs:361 (connect), :363 (every block RPC: data_timeout_ms)
    int64_t rpc_timeout_ms = 120 * 1000;   // parsed for compatibility; block RPCs use data_timeout_ms (block_client.rs:56)
    int64_t data_timeout_ms = 120 * 1000;
    bool enable_block_conn_pool = true;
    int64_t block_conn_idle_size = 128;       // idle connections kept by the pool, over ALL workers (block_client_pool.rs:147-155)
    int64_t block_conn_idle_time_ms = 60000;  // "block_conn_idle_time", DurationUnit string, default "60s" (client_conf.rs:412-413)
    int64_t failed_worker_ttl_ms = 10 * 60 * 1000;  // "failed_worker_ttl", DurationUnit string, default "10m" (client_conf.rs:139-141,374)
    std::string hostname;  // CURVINE_CLIENT_HOSTNAME override; default gethostname()
    Err init();            // client_conf.rs:228-281
};

// [b200] section: the GPU ingest pipeline (no reference counterpart)
struct B200Conf {
    int device = 0;
    int fetch_threads = 16;       // host threads pulling blocks into pinned slots
    int pinned_slots = 32;        // ring depth (slots of max block bytes + frame overhead)
    int verify_poly = 1;          // 0 = CRC-32 (reference tools), 1 = CRC-32C (north_star)
    bool verify = true;           // compare per-block CRC with the manifest on the GPU
    int verify_batch = 16;        // blocks per CRC launch
    int copy_streams = 1;         // H2D streams shared by the fetch threads (1 measured best on B200: no channel switching)
    int copy_group = 8;           // consecutive blocks moved by one cudaMemcpyAsync (bigger copies: closer to PCIe peak)
    int64_t gpu_chunk_size = 4 << 20;  // Running-request chunk for the framed GPU path (<= 16 MiB frame cap)
    bool zero_copy = false;       // short-circuit reads: DMA straight from cudaHostRegister'ed mmaps of the block files
    int64_t register_cache = 64ll << 30;  // bytes of registered mappings kept across calls (LRU)
    int64_t register_min_age_ms = 5000;   // "register_min_age" (duration string): a cached mapping used more recently than this is not
                                          // displaced by a newcomer (scan resistance); 0 = plain LRU
    int register_threads = 16;    // background registrar threads (a cold group goes through the pinned ring meanwhile); 0 = register inline
    bool register_when_idle = true;  // registrar threads yield to reads in flight (a cold pass runs at ring speed; mappings are
                                     // registered between reads); false = register concurrently with the cold pass
    bool arena = true;            // short-circuit Opens say accept_arena: arena-backed mem-tier blocks are DMA'd straight out of the
                                  // worker's arena segments (arena.h), which this context maps and pins once per segment
    std::vector<std::string> arena_dirs;  // "arena_preregister": worker data dirs (as in [worker] data_dir, tag optional) whose arena
                                          // segments are mapped + pinned in the background from the first device read (or
                                          // cv_fs_preregister) on -- off the read path; other segments are pinned when first met
    int64_t arena_register_slice = 256ll << 20;  // one cudaHostRegister call covers this much of a segment (slices go to register_threads)
    bool local_unix_socket = false;  // block connections to a worker on this host use its abstract unix socket (net.h) instead of loopback TCP
    int64_t socket_buffer = 0;       // explicit SO_RCVBUF/SO_SNDBUF for block connections (0 = kernel autotuning)
    bool gds = true;              // "gds" = "off" | "auto" (default): with auto, short-circuit reads of SSD/HDD/DISK-tier blocks go through
                                  // cuFileRead (gds.h) straight into HBM where GPUDirect Storage (nvidia-fs) is loaded; anything GDS
                                  // cannot serve goes through the pinned ring
    int numa_node = -1;           // bind fetch threads to this node's CPUs (-1: the GPU's node if discoverable, -2: no binding)
};

struct ClusterConf {
    ClientConf client;
    B200Conf b200;
    std::string cluster_id = "curvine";
    std::string namespace_manifest;        // file -> blocks table (stands in for master GetBlockLocations)
    std::vector<std::string> worker_dirs;  // worker.data_dir entries, e.g. "[MEM]/dev/shm/cv"
    std::string worker_hostname = "localhost";
    int worker_port = 0;
    bool worker_enable_send_file = true;
    bool worker_mem_arena = false;             // [worker] mem_arena: every [MEM] data dir keeps its blocks in one arena (arena.h)
    int64_t worker_arena_segment = 1ll << 30;  // [worker] arena_segment
    std::vector<int> worker_arena_numa;        // [worker] arena_numa = [node per MEM dir]
    int64_t worker_arena_reuse_delay_ms = 1000;  // [worker] arena_reuse_delay (duration string)
    int64_t worker_hbm_capacity = 0;     // [worker] hbm_capacity: bytes of device memory the HBM tier may hold (0 = unbounded, manual loads)
    int worker_hbm_promote_after = 0;    // [worker] hbm_promote_after: framed reads of a block before it is loaded into the tier (0 = never)
    int worker_hbm_device = 0;           // [worker] hbm_device

    static Err from_file(const std::string& path, ClusterConf* out);
    static Err from_string(const std::string& toml, ClusterConf* out);
};

// "128KB" -> 131072; plain integers pass through
Err parse_byte_size(const std::string& s, int64_t* out);
// DurationUnit::from_str (orpc/src/common/duration_unit.rs:66-108): "60s" "5m" "2h" "1d" "250ms" "250" (= ms) "1.5s" -> milliseconds
Err parse_duration_ms(const std::string& s, int64_t* out);

}  // namespace cv
