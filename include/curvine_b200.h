/*
 * curvine_b200.h -- upper boundary: the reader surface a Curvine client binds to (C ABI).
 *
 * Drop-in for the reference's reader path only.  Semantics, ownership, error and threading conventions are
 * the reference's own FFI conventions (curvine-libsdk, paths relative to /root/reference):
 *   handles      opaque pointers (Box::into_raw as i64: orpc/src/sys/ffi_utils.rs:47-49,64-66)
 *   errors       0 == SUCCESS (curvine-libsdk/src/java/mod.rs:23); failure returns -(ErrorKind)
 *                (curvine-common/src/error/fs_error.rs:35-66,324-326); EOF is not an error (length 0)
 *   cv_read      (address,length) of a buffer OWNED BY THE READER, valid until the next read/seek/close on
 *                that handle (curvine-libsdk/src/java/java_abi.rs:128-142, lib_fs_reader.rs:49-53)
 *   threading    a filesystem handle is shareable; a reader handle is single-threaded, no internal locking
 *                (lib_filesystem.rs:25-40); every call blocks
 * Entry point <- reference interface it replaces:
 *   cv_fs_new / cv_fs_close      LibFilesystem::new / closeFilesystem      curvine-libsdk/src/lib_filesystem.rs:25-40
 *   cv_open                      FileSystem::open -> Reader                curvine-common/src/fs/filesystem.rs:35,
 *                                                                          java_abi.rs:110-125
 *   cv_read                      Reader::blocking_read (read_chunk(None))  curvine-common/src/fs/reader.rs:84-88
 *   cv_read_buf / cv_read_full   Reader::read / Reader::read_full          reader.rs:71-81,126-141
 *   cv_fuse_read                 Reader::fuse_read                         reader.rs:101-124
 *   cv_seek / cv_pos / cv_len    Reader::seek / pos / len                  reader.rs:23-48, fs_reader.rs:109-126
 *   cv_close_reader              Reader::complete + drop                   java_abi.rs:157-166
 *   cv_read_device, cv_read_device_sharded, cv_read_many_device, cv_verify, cv_fuse_read_device
 *                                the CUDA counterpart the north_star adds behind the same reader handle
 *                                (no reference counterpart: the reference has no GPU code)
 * The cv_worker_* and cv_synth_* entry points are the test/bench fixture (the analogue of the reference's
 * in-process MiniCluster + Worker::start_standalone, curvine-server/tests/worker_test.rs:35-48); they are not
 * part of the drop-in surface.
 */
#ifndef CURVINE_B200_H
#define CURVINE_B200_H

#include <stddef.h>
#include <stdint.h>

#include "curvine_b200_kernels.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cv_fs cv_fs;
typedef struct cv_reader cv_reader;
typedef struct cv_worker cv_worker;
typedef struct cv_writer cv_writer;

/* -(ErrorKind) values a caller is likely to test for (fs_error.rs:35-66) */
#define CV_OK 0
#define CV_ERR_IO (-1)
#define CV_ERR_TIMEOUT (-4)
#define CV_ERR_PB_DECODE (-5)
#define CV_ERR_FILE_NOT_FOUND (-8)
#define CV_ERR_ABNORMAL_DATA (-12)
#define CV_ERR_UNSUPPORTED (-19)
#define CV_ERR_COMMON (-10000)

/* Message of the last failure on the calling thread ("" if none). */
const char* cv_last_error(void);
void cv_free(void* p);

/* ---- filesystem handle: conf (TOML subset: [client] read knobs with the reference's names and defaults,
 *      [worker], [b200]) + the file->blocks namespace (stand-in for master GetBlockLocations) */
int64_t cv_fs_new(const char* conf_path, cv_fs** out);
int64_t cv_fs_new_from_string(const char* conf_toml, cv_fs** out);
int64_t cv_fs_load_namespace(cv_fs* fs, const char* manifest_path);
int64_t cv_fs_load_namespace_string(cv_fs* fs, const char* manifest_text);
/* Drops the handle's reference to the filesystem context.  Readers / writers opened from it hold their own (as FsReader holds an
 * Arc<FsContext> in the reference): they stay valid and must still be closed; the context and its GPU pipeline go with the last holder. */
int64_t cv_fs_close(cv_fs* fs);
/* Block until everything this context pins in the background is pinned: the arena segments queued by cv_fs_preregister / the
 * first device read (mem-arena tier), and -- for the reference's one-file-per-block mem tier -- the registrar's mmap +
 * cudaHostRegister of block files seen by earlier device reads.  Optional: a read that needs an arena segment whose pinning is
 * still in progress waits for that one segment; a block FILE that is not registered yet goes through the pinned ring (by
 * default, [b200] register_when_idle = true, the registrar only works while no device read is in flight). */
int64_t cv_fs_wait_registered(cv_fs* fs);
/* Mem-arena tier (worker `[worker] mem_arena = true`, curvine_b200/csrc/host/arena.h): start mapping + pinning the arena
 * segments of the dirs named in `[b200] arena_preregister` now, in the background ("mount time"; otherwise it starts with
 * the first device read).  cv_fs_wait_registered waits for it.  Once a segment is pinned, every block the worker keeps in
 * it -- of any file, written at any time -- is DMA'd straight out of it: the first read of a file costs what a re-read costs.
 * stats: out[0]=segments mapped, out[1]=bytes pinned, out[2]=registration wall time (us), out[3]=block jobs and out[4]=bytes
 * DMA'd straight out of pinned segments. */
int64_t cv_fs_preregister(cv_fs* fs);
int64_t cv_fs_arena_stats(cv_fs* fs, uint64_t out[5]);
/* client metrics (client_metrics.rs:24-35): out[0]=read_bytes out[1]=read_time_us */
int64_t cv_fs_metrics(cv_fs* fs, int64_t out[2]);
/* block connection pool (block_client_pool.rs:102-168): out[0]=idle connections now (idle_conn), out[1]=connections opened so far,
 * out[2]=pooled connections dropped because they sat idle for block_conn_idle_time or longer */
int64_t cv_fs_pool_stats(cv_fs* fs, int64_t out[3]);

/* ---- reader */
int64_t cv_open(cv_fs* fs, const char* path, cv_reader** out, int64_t* len);
int64_t cv_read(cv_reader* r, const uint8_t** ptr, int64_t* len);
int64_t cv_read_buf(cv_reader* r, uint8_t* buf, int64_t cap, int64_t* n);
int64_t cv_read_full(cv_reader* r, uint8_t* buf, int64_t cap, int64_t* n);
/* seek(pos) then whole chunks until len bytes: payload copied to buf, chunk boundaries to seg_lens[0..*n_segs) */
int64_t cv_fuse_read(cv_reader* r, int64_t pos, int64_t len, uint8_t* buf, int64_t* n, int64_t* seg_lens,
                     int32_t max_segs, int32_t* n_segs);
int64_t cv_seek(cv_reader* r, int64_t pos);
int64_t cv_pos(cv_reader* r);
int64_t cv_len(cv_reader* r);
int64_t cv_chunk_size(cv_reader* r);
int64_t cv_close_reader(cv_reader* r);

/* ---- CUDA counterpart (same handle, same pos).  d_dst is device memory; work is ordered on `stream`. */
int64_t cv_read_device(cv_reader* r, void* d_dst, int64_t cap, cv_stream_t stream, int64_t* nbytes);
/* blocks b with b % world == rank, back to back in block_size slots (slot j = block j*world+rank) */
int64_t cv_read_device_sharded(cv_reader* r, int32_t rank, int32_t world, void* d_dst, int64_t cap,
                               cv_stream_t stream, int64_t* nbytes);
/* Small-file batching (config C5): n whole files in ONE pipelined pass; file i lands at d_dst + dst_offs[i].
 * Open/Complete RPCs, H2D copies and CRC launches of all files overlap; returns after verification
 * (sum_crc / n_bad / n_verified as in cv_verify).  Replaces n x (FileSystem::open + Reader::fuse_read + complete). */
int64_t cv_read_many_device(cv_fs* fs, const char* const* paths, int32_t n, void* d_dst, const int64_t* dst_offs, int64_t cap,
                            cv_stream_t stream, uint64_t* sum_crc, uint32_t* n_bad, uint64_t* n_verified, int64_t* total_bytes);
/* The plan cv_read_device_sharded executes (host-only, no GPU needed): for i < *n, block_index[i] of the file starts
 * at file_off[i], is len[i] bytes long and lands at dst_off[i] = i * block_size.  Arrays may be NULL; cap = their length. */
int64_t cv_shard_plan(cv_reader* r, int32_t rank, int32_t world, int64_t* block_index, int64_t* file_off, int64_t* len,
                      int64_t* dst_off, int32_t cap, int32_t* n, int64_t* total_bytes);
/* FUSE-shaped device read: seek(pos), read len bytes into HBM scratch, then scatter them into n_pages page
 * buffers (d_page_base + page_offsets[i], page_size each; last one partial) with the K3 gather kernel. */
int64_t cv_fuse_read_device(cv_reader* r, int64_t pos, int64_t len, void* d_scratch, void* d_page_base,
                            const uint64_t* page_offsets, int32_t n_pages, int64_t page_size, cv_stream_t stream,
                            int64_t* nbytes);
/* One small file, one call: open -> fuse-shaped device read of the first `len` bytes -> CRC verify -> close.  Blocks until the
 * pages hold the bytes; *n_bad = blocks whose CRC differs from the manifest. */
int64_t cv_fuse_read_file_device(cv_fs* fs, const char* path, int64_t len, void* d_scratch, void* d_page_base,
                                 const uint64_t* page_offsets, int32_t n_pages, int64_t page_size, cv_stream_t stream,
                                 int64_t* nbytes, uint32_t* n_bad);
/* Blocks until outstanding device reads of this handle finished.  sum_crc = u64 sum of per-block CRCs of every
 * whole block read so far; n_bad = blocks whose CRC differs from the manifest; n_verified = blocks compared. */
int64_t cv_verify(cv_reader* r, uint64_t* sum_crc, uint32_t* n_bad, uint64_t* n_verified);

typedef struct CvReadStats {
    uint64_t bytes, blocks, verified, h2d_bytes, kernel_launches;
    double fetch_sec, wall_sec;
    uint64_t reg_hits, reg_misses; /* registered-mapping cache of the zero-copy path */
    double ring_alloc_sec;         /* one-off pinned-ring allocation time of the context (first cold read pays it) */
    uint64_t reg_rejected;         /* mappings not admitted: the cache was full of in-use or recently used ones */
    uint64_t reg_bytes;            /* bytes registered through the cache right now (<= register_cache) */
    uint64_t gds_bytes;            /* bytes read file -> HBM by cuFileRead (disk tiers, [b200] gds) */
} CvReadStats;
/* GPUDirect Storage probe: out[0] = 1 when libcufile loaded and its driver opened, out[1] = 1 when the nvidia-fs kernel module is
 * not loaded (cuFile would only have its compatibility mode, which is not used: libcufile is not loaded and out = {0, 1}).  The
 * message (cv_last_error) carries the detail either way. */
int64_t cv_gds_info(int64_t out[2]);
int64_t cv_device_stats(cv_reader* r, CvReadStats* out);

/* ---- write-side mirror ("next" row 8f-1): WriteBlock = 80, Open -> Running x N -> Complete per block
 * (curvine-client/src/block/block_writer_remote.rs:36-140, block_client.rs:97-219; worker write_handler.rs:90-300).
 * Blocks of block_size are allocated one after another (block_id = inode<<24 | seq); per-block CRC-32/CRC-32C are
 * computed at write time and land in the manifest, so a later cv_verify compares read-side with write-side CRCs.
 * cv_write takes host bytes; cv_write_device takes HBM bytes: K4 (cvk_pack_frames) writes the request prefixes, copies the
 * payload behind them and CRCs the source in one pass, the wire image goes D2H once and onto the socket verbatim.
 * cv_writer_close(cancel=0) commits and registers the file in the filesystem handle's namespace (manifest text returned,
 * cv_free); cancel=1 aborts the open block. */
int64_t cv_writer_open(cv_fs* fs, const char* path, int64_t inode_id, int64_t block_size, int32_t storage_type,
                       const char* worker_host, int32_t worker_port, int64_t chunk_size, cv_writer** out);
int64_t cv_write(cv_writer* w, const uint8_t* buf, int64_t n);
int64_t cv_write_device(cv_writer* w, const void* d_src, int64_t n, cv_stream_t stream);
int64_t cv_writer_close(cv_writer* w, int32_t cancel, char** manifest_out);

/* ---- fixture: in-process worker over a BlockStore directory tree + synthetic files */
int64_t cv_worker_start(const char* conf_toml, cv_worker** out, int32_t* port);
int64_t cv_worker_stop(cv_worker* w);
/* HBM as a worker tier ("next" row 8f-2): copy a finalized block into device memory; from then on REMOTE reads of it are
 * served from HBM as frames packed on the GPU (K4) -- the block file is no longer touched.
 * stats: out[0]=resident blocks [1]=reads served from HBM [2]=payload bytes packed by K4. */
int64_t cv_worker_hbm_load(cv_worker* w, int64_t block_id, int32_t device);
int64_t cv_worker_hbm_stats(cv_worker* w, int64_t out[3]);
/* Promotion into the tier is asynchronous (a promoter thread; the read that crossed hbm_promote_after is served from the store):
 * wait until nothing is queued or running. */
int64_t cv_worker_hbm_drain(cv_worker* w);
/* HBM tier occupancy and policy counters ([worker] hbm_capacity / hbm_promote_after / hbm_device): out[0]=resident blocks,
 * out[1]=resident bytes, out[2]=capacity (0 = unbounded), out[3]=evictions (LRU, never a block that is being read),
 * out[4]=promotions (blocks loaded because they were read remotely hbm_promote_after times), out[5]=refused loads */
int64_t cv_worker_hbm_tier(cv_worker* w, int64_t out[6]);
/* out[0]=read_bytes [1]=read_time_us [2]=read_count [3]=read_blocks{local} [4]=read_blocks{remote} [5]=num_blocks */
int64_t cv_worker_metrics(cv_worker* w, int64_t out[6]);
/* Write `len` bytes of synthetic content as blocks of `block_size` into the worker's BlockStore (reference
 * layout) and return the manifest text (malloc'd, cv_free) with per-block CRC-32 / CRC-32C.
 * mode 0: xoshiro256** per block (SURVEY.md 8d); mode 1: "az" repeated lowercase buffer; mode 2: every
 * hole_every-th block is a hole (no file, no location). */
int64_t cv_synth_create_file(cv_worker* w, const char* path, int64_t inode_id, int64_t len, int64_t block_size,
                             int32_t storage_type, int32_t mode, int32_t hole_every, int32_t threads,
                             const char* worker_hostname, char** manifest_out);
/* Remove the n_blocks blocks of synthetic file `inode_id` from the worker's BlockStore (files unlinked / arena extents freed). */
int64_t cv_synth_delete_file(cv_worker* w, int64_t inode_id, int64_t n_blocks);
/* Mem arenas of the worker: out[0]=arena dirs, out[1]=segments, out[2]=segment bytes, out[3]=bytes in use,
 * out[4]=time spent creating + populating the segments (us). */
int64_t cv_worker_arena_stats(cv_worker* w, int64_t out[5]);
/* NUMA-aware mem-tier placement for round-robin shards: after cv_synth_set_shard_world(G), block b of newly created
 * files is first-touched on the NUMA node of GPU b % G (G = 1: everything next to GPU 0; 0 turns it off), and goes to the
 * (b % G)-th data dir of its storage type -- with one [MEM] arena dir per GPU, GPU g's blocks all live in arena g. */
int64_t cv_synth_set_shard_world(int32_t shard_world);
/* NUMA node of the PCIe root CUDA device `device` hangs off, -1 when unknown ([worker] arena_numa, [b200] numa_node). */
int64_t cv_gpu_numa_node(int32_t device);
/* fill buf with block `block_index` of file `file_id` (mode 0 generator) */
void cv_synth_block(uint64_t file_id, uint64_t block_index, uint8_t* buf, size_t len);
/* host CRC used for manifests (slicing / SSE4.2) */
uint32_t cv_host_crc(int poly, const uint8_t* buf, size_t len);

#ifdef __cplusplus
}
#endif
#endif
