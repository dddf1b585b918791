#include "gpu_reader.h"

#include <cuda_runtime.h>
#include <errno.h>
#include <fcntl.h>
#include <sched.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <deque>
#include <list>
#include <set>

#include <fstream>

#include "../../../include/curvine_b200_kernels.h"
#include "block_store.h"
#include "gds.h"
#include "net.h"

namespace cv {

#define CU_TRY(x)                                                                                   \
    do {                                                                                            \
        cudaError_t e_ = (x);                                                                       \
        if (e_ != cudaSuccess) return Err::io(str_printf("%s: %s", #x, cudaGetErrorString(e_)));    \
    } while (0)
#define CVK_TRY(x)                                                                                  \
    do {                                                                                            \
        int e_ = (x);                                                                               \
        if (e_ != 0) return Err::io(str_printf("%s: %s", #x, cudaGetErrorString(cudaError_t(e_)))); \
    } while (0)

// ------------------------------------------------------------------ registered mem-tier mappings (zero-copy ingest)
//
// A mem-tier block file lives in tmpfs page-cache pages.  Instead of pread()ing it into a pinned slot (one CPU copy
// per byte), map the block files of one copy group back to back into a reserved VA range, cudaHostRegister the range
// once, and let the copy engine DMA straight out of the page cache.  Mappings are cached (LRU by bytes, never more than
// `register_cache` bytes registered through the cache) and revalidated by (inode, size, mtime) on every use; block files
// are write-once in Curvine.
// Admission is scan-resistant: a new mapping only displaces mappings that nobody is using AND that have not been used for
// `register_min_age` (default 5 s); otherwise the newcomer is not cached (its group keeps going through the pinned ring).
// With plain LRU a sequential re-read of a file larger than the cache finds every group evicted just before it gets there
// -- 0 hits while paying registration every pass; with this rule the first cache-full of groups stays registered and a
// cyclic scan hits cache/working-set of the time, while a working set that moved away ages out after register_min_age.
struct RegMapping {
    std::string key;
    uint8_t* base = nullptr;
    size_t bytes = 0;     // registered extent (page-rounded)
    std::vector<uint64_t> stamps;  // inode, size, mtime_ns per member file
    bool registered = false;
    double last_used = 0;  // now_sec() of the last find() hit or the insertion (under RegCache's lock)
    ~RegMapping() {
        if (registered) cudaHostUnregister(base);
        if (base) munmap(base, bytes);
    }
};

class RegCache {
   public:
    size_t capacity = 0;   // bytes; 0 disables caching (mappings live for one call)
    double min_age_sec = 5.0;  // a mapping used more recently than this is not displaced by a newcomer
    std::shared_ptr<RegMapping> find(const std::string& key, const std::vector<uint64_t>& stamps) {
        std::shared_ptr<RegMapping> stale;  // destroyed (unregistered, unmapped) outside the lock
        std::lock_guard<std::mutex> lk(mu_);
        auto it = map_.find(key);
        if (it == map_.end()) return nullptr;
        if (it->second->second->stamps != stamps) {  // file replaced: drop the stale mapping
            stale = it->second->second;
            bytes_ -= stale->bytes;
            lru_.erase(it->second);
            map_.erase(it);
            return nullptr;
        }
        lru_.splice(lru_.begin(), lru_, it->second);
        it->second->second->last_used = now_sec();
        hits++;
        return it->second->second;
    }
    // -> true when the mapping was admitted.  A rejected mapping stays valid for the caller's own use and goes away with it.
    bool insert(const std::shared_ptr<RegMapping>& m) {
        std::vector<std::shared_ptr<RegMapping>> evicted;  // destroyed outside the lock
        std::lock_guard<std::mutex> lk(mu_);
        if (capacity == 0 || m->bytes > capacity) return false;
        auto dup = map_.find(m->key);
        if (dup != map_.end()) {  // same group registered twice (two contexts' worth of threads raced): the newer one wins
            bytes_ -= dup->second->second->bytes;
            evicted.push_back(dup->second->second);
            lru_.erase(dup->second);
            map_.erase(dup);
        }
        const double now = now_sec();
        // make room from the cold end; stop at the first entry that is in use or still young
        while (bytes_ + m->bytes > capacity && !lru_.empty()) {
            auto& back = lru_.back();
            if (back.second.use_count() > 1 || now - back.second->last_used < min_age_sec) break;
            bytes_ -= back.second->bytes;
            evicted.push_back(back.second);
            map_.erase(back.first);
            lru_.pop_back();
        }
        if (bytes_ + m->bytes > capacity) {
            rejected++;
            return false;
        }
        m->last_used = now;
        lru_.emplace_front(m->key, m);
        map_[m->key] = lru_.begin();
        bytes_ += m->bytes;
        return true;
    }
    // would insert() admit a mapping of `bytes` right now?  (asked BEFORE paying for mmap + cudaHostRegister)
    bool can_admit(size_t bytes) {
        std::lock_guard<std::mutex> lk(mu_);
        if (capacity == 0 || bytes > capacity) return false;
        size_t room = capacity - std::min(capacity, bytes_);
        const double now = now_sec();
        for (auto it = lru_.rbegin(); room < bytes && it != lru_.rend(); ++it) {
            if (it->second.use_count() > 1 || now - it->second->last_used < min_age_sec) break;
            room += it->second->bytes;
        }
        return room >= bytes;
    }
    void clear() {
        std::lock_guard<std::mutex> lk(mu_);
        map_.clear();
        lru_.clear();
        bytes_ = 0;
    }
    size_t bytes() {
        std::lock_guard<std::mutex> lk(mu_);
        return bytes_;
    }
    std::atomic<uint64_t> hits{0}, misses{0}, rejected{0};

   private:
    std::mutex mu_;
    std::list<std::pair<std::string, std::shared_ptr<RegMapping>>> lru_;
    std::unordered_map<std::string, std::list<std::pair<std::string, std::shared_ptr<RegMapping>>>::iterator> map_;
    size_t bytes_ = 0;
};

// Map `paths` (lens[i] bytes each; all but the last a multiple of the page size) contiguously and register the range.
static Err map_and_register(const std::vector<std::string>& paths, const std::vector<int64_t>& lens, std::shared_ptr<RegMapping>* out,
                            std::vector<uint64_t>* stamps_out) {
    const size_t page = 4096;
    size_t total = 0;
    for (size_t i = 0; i < paths.size(); i++) {
        if (i + 1 < paths.size() && lens[i] % static_cast<int64_t>(page)) return Err::common("block length is not page aligned");
        total += (static_cast<size_t>(lens[i]) + page - 1) / page * page;
    }
    std::shared_ptr<RegMapping> m(new RegMapping());
    void* base = mmap(nullptr, total, PROT_NONE, MAP_PRIVATE | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
    if (base == MAP_FAILED) return Err::io(str_printf("mmap reserve: %s", strerror(errno)));
    m->base = static_cast<uint8_t*>(base), m->bytes = total;
    size_t off = 0;
    for (size_t i = 0; i < paths.size(); i++) {
        // cudaHostRegister needs a writable shared mapping here (cudaHostRegisterReadOnly is not supported on this
        // platform); nothing ever writes through it.  Read-only block files fall back to the pinned ring.
        const int fd = ::open(paths[i].c_str(), O_RDWR | O_CLOEXEC);
        if (fd < 0) return Err(kUnsupported, str_printf("open %s read-write: %s", paths[i].c_str(), strerror(errno)));
        struct stat st;
        fstat(fd, &st);
        if (st.st_size < lens[i]) {
            ::close(fd);
            return Err::io("block file shorter than the block length");
        }
        m->stamps.push_back(static_cast<uint64_t>(st.st_ino)), m->stamps.push_back(static_cast<uint64_t>(st.st_size));
        m->stamps.push_back(static_cast<uint64_t>(st.st_mtim.tv_sec) * 1000000000ull + static_cast<uint64_t>(st.st_mtim.tv_nsec));
        const size_t span = (static_cast<size_t>(lens[i]) + page - 1) / page * page;
        void* p = mmap(m->base + off, span, PROT_READ | PROT_WRITE, MAP_SHARED | MAP_FIXED | MAP_POPULATE, fd, 0);
        ::close(fd);
        if (p == MAP_FAILED) return Err::io(str_printf("mmap %s: %s", paths[i].c_str(), strerror(errno)));
        off += span;
    }
    cudaError_t e = cudaHostRegister(m->base, total, cudaHostRegisterDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return Err(kUnsupported, str_printf("cudaHostRegister(%zu): %s", total, cudaGetErrorString(e)));
    }
    m->registered = true;
    *stamps_out = m->stamps;
    *out = std::move(m);
    return Err::ok();
}

static bool stat_stamps(const std::vector<std::string>& paths, std::vector<uint64_t>* stamps) {
    stamps->clear();
    for (const auto& p : paths) {
        struct stat st;
        if (stat(p.c_str(), &st) != 0) return false;
        stamps->push_back(static_cast<uint64_t>(st.st_ino)), stamps->push_back(static_cast<uint64_t>(st.st_size));
        stamps->push_back(static_cast<uint64_t>(st.st_mtim.tv_sec) * 1000000000ull + static_cast<uint64_t>(st.st_mtim.tv_nsec));
    }
    return true;
}

// Background registration: a cache miss does not stall the read.  The foreground moves the group through the pinned
// ring right away (cold pass at ring speed) while a few registrar threads mmap + cudaHostRegister the same files so that
// the NEXT pass over them is zero-copy.  cudaHostRegister pins 4 KiB pages at ~13-26 GB/s on the B200 box and
// serialises with copy enqueues inside the driver, so by default (`register_when_idle`) the registrar threads yield to
// reads in flight: `hold` counts them, and a registrar only starts a new group while it is zero (or while a caller is
// blocked in drain()).
class Registrar {
   public:
    struct Job {
        std::string key;
        std::vector<std::string> paths;
        std::vector<int64_t> lens;
    };
    void start(int threads, int device, RegCache* cache, std::vector<int> cpus, const std::atomic<int>* hold) {
        device_ = device, cache_ = cache, cpus_ = std::move(cpus), hold_ = hold;
        for (int t = 0; t < threads; t++) threads_.emplace_back([this] { loop(); });
    }
    void submit(Job j) {
        std::lock_guard<std::mutex> lk(mu_);
        if (stop_ || unsupported.load() || !pending_keys_.insert(j.key).second) return;
        q_.push_back(std::move(j));
        cv_.notify_one();
    }
    void stop() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
            q_.clear();
            cv_.notify_all();
        }
        for (auto& t : threads_) t.join();
        threads_.clear();
    }
    void drain() {  // wait until the queue is empty and no registration is in flight
        std::unique_lock<std::mutex> lk(mu_);
        draining_++;
        idle_cv_.wait(lk, [&] { return (q_.empty() && busy_ == 0) || stop_; });
        draining_--;
    }
    size_t backlog() {
        std::lock_guard<std::mutex> lk(mu_);
        return q_.size() + static_cast<size_t>(busy_);
    }
    std::atomic<bool> unsupported{false};
    std::atomic<uint64_t> registered{0};

   private:
    void loop() {
        if (!cpus_.empty()) {
            cpu_set_t set;
            CPU_ZERO(&set);
            for (int c : cpus_) CPU_SET(c, &set);
            sched_setaffinity(0, sizeof(set), &set);
        }
        cudaSetDevice(device_);
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
                if (stop_) return;
                if (hold_ && hold_->load(std::memory_order_acquire) > 0 && draining_ == 0) {  // a read is in flight: stay out of its way
                    lk.unlock();
                    usleep(300);
                    continue;
                }
                j = std::move(q_.front());
                q_.pop_front();
                busy_++;
            }
            std::shared_ptr<RegMapping> m;
            std::vector<uint64_t> stamps;
            size_t job_bytes = 0;
            for (int64_t l : j.lens) job_bytes += (static_cast<size_t>(l) + 4095) / 4096 * 4096;
            Err e = cache_->can_admit(job_bytes) ? map_and_register(j.paths, j.lens, &m, &stamps) : Err(kCommon, "registration cache is full");
            if (!e) {
                m->key = j.key;
                if (cache_->insert(m)) registered++;
            } else if (e.kind == kUnsupported) {
                unsupported.store(true);
            }
            std::lock_guard<std::mutex> lk(mu_);
            pending_keys_.erase(j.key);
            busy_--;
            if (q_.empty() && busy_ == 0) idle_cv_.notify_all();
        }
    }
    int device_ = 0;
    RegCache* cache_ = nullptr;
    std::vector<int> cpus_;
    std::vector<std::thread> threads_;
    std::mutex mu_;
    std::condition_variable cv_, idle_cv_;
    std::deque<Job> q_;
    std::set<std::string> pending_keys_;
    int busy_ = 0, draining_ = 0;
    bool stop_ = false;
    const std::atomic<int>* hold_ = nullptr;
};

// ------------------------------------------------------------------ mem-arena segments (pinned once, off the read path)
//
// An arena-backed worker (arena.h) keeps every mem-tier block as an extent of a few large tmpfs segment files.  A segment is
// mapped and cudaHostRegister'ed ONCE per context -- in the background from the first device read on for the dirs named in
// `[b200] arena_preregister`, on demand for any other segment an Open names -- and stays pinned until the context closes.
// From then on every block in it, whatever file it belongs to and whenever it was written, is DMA'd straight out of the
// segment: no per-file or per-block client state, so the first read of a file runs at the same rate as a re-read.
// Registration is sliced (`arena_register_slice`) so that all registrar threads pin one segment together.
struct ArenaSeg {
    std::string path;
    uint8_t* base = nullptr;
    size_t bytes = 0, slice = 0;
    uint64_t ino = 0;
    std::vector<uint8_t> slice_registered;
    std::mutex mu;
    std::condition_variable cv;
    size_t slices_left = 0;
    bool done = false;
    Err err;
    ~ArenaSeg() {
        if (base) mprotect(base, bytes, PROT_READ | PROT_WRITE);
        for (size_t i = 0; i < slice_registered.size(); i++)
            if (slice_registered[i]) cudaHostUnregister(base + i * slice);
        if (base) munmap(base, bytes);
    }
};

class ArenaSegs {
   public:
    std::atomic<uint64_t> dma_jobs{0}, dma_bytes{0};  // block jobs / bytes moved straight out of a pinned segment
    std::atomic<bool> unsupported{false};             // cudaHostRegister refuses these mappings: arena blocks go through the ring
    double register_sec = 0;                          // wall time from the first slice queued to the last one pinned (under mu_)

    void start(int threads, int device, std::vector<int> cpus, size_t slice) {
        device_ = device, cpus_ = std::move(cpus), slice_ = std::max<size_t>(slice, 2 << 20) & ~size_t(4095);
        for (int t = 0; t < std::max(1, threads); t++) threads_.emplace_back([this] { loop(); });
    }
    void stop() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
            q_.clear();
            cv_.notify_all();
        }
        for (auto& t : threads_) t.join();
        threads_.clear();
        std::lock_guard<std::mutex> lk(mu_);
        segs_.clear();
        retired_.clear();
    }
    // Every seg_* file under <data_dir>/<cluster_id>/arena is queued for mapping + pinning.  Returns immediately.
    void preregister_dir(const std::string& arena_dir) {
        for (int k = 0;; k++) {
            const std::string p = str_printf("%s/seg_%04d", arena_dir.c_str(), k);
            struct stat st;
            if (stat(p.c_str(), &st) != 0) break;
            std::shared_ptr<ArenaSeg> seg;
            begin(p, &seg);
        }
    }
    // The pinned mapping of segment `path` (blocks until it is fully registered; starts the registration if nobody has).
    Err get(const std::string& path, std::shared_ptr<ArenaSeg>* out) {
        std::shared_ptr<ArenaSeg> seg;
        CV_RETURN_IF_ERR(begin(path, &seg));
        std::unique_lock<std::mutex> lk(seg->mu);
        seg->cv.wait(lk, [&] { return seg->done; });
        if (seg->err) return seg->err;
        *out = std::move(seg);
        return Err::ok();
    }
    void drain() {  // wait until everything queued so far is pinned
        std::vector<std::shared_ptr<ArenaSeg>> all;
        {
            std::lock_guard<std::mutex> lk(mu_);
            for (auto& kv : segs_) all.push_back(kv.second);
        }
        for (auto& seg : all) {
            std::unique_lock<std::mutex> lk(seg->mu);
            seg->cv.wait(lk, [&] { return seg->done; });
        }
    }
    void stats(uint64_t* n_segs, uint64_t* bytes, double* sec) {
        std::lock_guard<std::mutex> lk(mu_);
        *n_segs = segs_.size(), *bytes = 0, *sec = register_sec;
        for (auto& kv : segs_) *bytes += kv.second->err ? 0 : kv.second->bytes;
    }

   private:
    Err begin(const std::string& path, std::shared_ptr<ArenaSeg>* out) {
        struct stat st;
        if (stat(path.c_str(), &st) != 0) return Err::io(str_printf("arena segment %s: %s", path.c_str(), strerror(errno)));
        std::lock_guard<std::mutex> lk(mu_);
        auto it = segs_.find(path);
        if (it != segs_.end() && it->second->ino == static_cast<uint64_t>(st.st_ino) && it->second->bytes == static_cast<size_t>(st.st_size)) {
            *out = it->second;
            return Err::ok();
        }
        if (it != segs_.end()) retired_.push_back(it->second);  // the file was replaced (worker restarted on a fresh dir): copies may still be in flight
        if (unsupported.load()) return Err(kUnsupported, "cudaHostRegister of arena segments is not supported here");
        std::shared_ptr<ArenaSeg> seg(new ArenaSeg());
        seg->path = path, seg->bytes = static_cast<size_t>(st.st_size), seg->ino = static_cast<uint64_t>(st.st_ino), seg->slice = slice_;
        // cudaHostRegister needs a writable shared mapping (cudaHostRegisterReadOnly is refused on this platform); the mapping is
        // write-protected again as soon as it is pinned
        const int fd = ::open(path.c_str(), O_RDWR | O_CLOEXEC);
        if (fd < 0) return Err(kUnsupported, str_printf("open %s read-write: %s", path.c_str(), strerror(errno)));
        void* m = mmap(nullptr, seg->bytes, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
        ::close(fd);
        if (m == MAP_FAILED) return Err::io(str_printf("mmap %s: %s", path.c_str(), strerror(errno)));
        seg->base = static_cast<uint8_t*>(m);
        const size_t n = (seg->bytes + slice_ - 1) / slice_;
        seg->slice_registered.assign(n, 0);
        seg->slices_left = n;
        if (busy_ == 0 && q_.empty()) t_first_ = now_sec();
        for (size_t i = 0; i < n; i++) q_.emplace_back(seg, i);
        segs_[path] = seg;
        cv_.notify_all();
        *out = std::move(seg);
        return Err::ok();
    }
    void loop() {
        if (!cpus_.empty()) {
            cpu_set_t set;
            CPU_ZERO(&set);
            for (int c : cpus_) CPU_SET(c, &set);
            sched_setaffinity(0, sizeof(set), &set);
        }
        cudaSetDevice(device_);
        for (;;) {
            std::pair<std::shared_ptr<ArenaSeg>, size_t> job;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
                if (stop_) return;
                job = std::move(q_.front());
                q_.pop_front();
                busy_++;
            }
            ArenaSeg& seg = *job.first;
            const size_t off = job.second * seg.slice, len = std::min(seg.slice, seg.bytes - off);
#ifdef MADV_POPULATE_WRITE
            // map the slice's (already allocated) tmpfs pages in bulk first: the page-by-page faults cudaHostRegister would
            // otherwise take on a fresh mapping are what made pinning 3x slower than on the mapping that created the pages
            madvise(seg.base + off, len, MADV_POPULATE_WRITE);
#endif
            const cudaError_t ce = cudaHostRegister(seg.base + off, len, cudaHostRegisterDefault);
            if (ce != cudaSuccess) cudaGetLastError();
            bool last = false;
            {
                std::lock_guard<std::mutex> lk(seg.mu);
                if (ce == cudaSuccess) seg.slice_registered[job.second] = 1;
                else if (!seg.err) seg.err = Err(kUnsupported, str_printf("cudaHostRegister(%s + %zu, %zu): %s", seg.path.c_str(), off, len, cudaGetErrorString(ce)));
                last = --seg.slices_left == 0;
                if (last) {
                    if (!seg.err) mprotect(seg.base, seg.bytes, PROT_READ);  // pinned pages stay DMA-able; nothing in this process can scribble on them
                    else unsupported.store(true);
                    seg.done = true;
                    seg.cv.notify_all();
                }
            }
            std::lock_guard<std::mutex> lk(mu_);
            busy_--;
            if (busy_ == 0 && q_.empty()) register_sec += now_sec() - t_first_;
        }
    }
    int device_ = 0;
    size_t slice_ = 256 << 20;
    std::vector<int> cpus_;
    std::vector<std::thread> threads_;
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<std::pair<std::shared_ptr<ArenaSeg>, size_t>> q_;
    std::unordered_map<std::string, std::shared_ptr<ArenaSeg>> segs_;
    std::vector<std::shared_ptr<ArenaSeg>> retired_;
    int busy_ = 0;
    double t_first_ = 0;
    bool stop_ = false;
};

// ------------------------------------------------------------------ GpuIngest: ring + streams

class GpuIngest {
   public:
    int device = 0;
    int nslots = 0;
    size_t slot_bytes = 0;
    uint8_t* pinned = nullptr;
    uint8_t* d_stage = nullptr;  // framed mode only
    size_t d_stage_bytes = 0;
    std::vector<cudaEvent_t> copy_ev, free_ev;
    std::vector<cudaStream_t> copy_streams;
    cudaStream_t vstream = nullptr;
    cudaEvent_t done_ev = nullptr;
    std::vector<int> cpus;
    std::mutex mu;  // one read_device at a time per context
    // per-call device tables + pinned result mirror, shared by every reader of the context
    uint8_t* d_tables = nullptr;
    size_t d_tables_cap = 0;
    uint8_t* h_result = nullptr;
    size_t h_result_cap = 0;
    uint8_t* h_tables = nullptr;  // pinned image of the per-call tables (off/len/expect/skip, stream descriptors): uploads are truly
    size_t h_tables_cap = 0;      // asynchronous, nothing waits for them (a pageable source makes cudaMemcpyAsync drain the stream first)
    GpuFsReader* pending_owner = nullptr;  // reader whose results still sit in h_result
    RegCache reg;
    Registrar registrar;
    ArenaSegs arena;
    cudaEvent_t entry_ev = nullptr;  // what the caller's stream had queued when a read started
    bool register_inline = false;
    std::atomic<int> reads_in_flight{0};  // run_jobs calls between entry and return (the registrar yields to them)
    double ring_alloc_sec = 0;            // time spent allocating the pinned ring (one-off per context and slot size)

    Err ensure_tables(size_t tables_bytes, size_t result_bytes) {
        if (tables_bytes > d_tables_cap) {
            if (d_tables) cudaFree(d_tables);
            d_tables_cap = tables_bytes * 2;
            CU_TRY(cudaMalloc(&d_tables, d_tables_cap));
        }
        if (tables_bytes > h_tables_cap) {
            if (h_tables) cudaFreeHost(h_tables);
            h_tables_cap = tables_bytes * 2;
            CU_TRY(cudaHostAlloc(&h_tables, h_tables_cap, cudaHostAllocDefault));
        }
        if (result_bytes > h_result_cap) {
            if (h_result) cudaFreeHost(h_result);
            h_result_cap = result_bytes * 2;
            CU_TRY(cudaHostAlloc(&h_result, h_result_cap, cudaHostAllocDefault));
        }
        return Err::ok();
    }

    Err init(const B200Conf& c) {
        device = c.device;
        CU_TRY(cudaSetDevice(device));
        CVK_TRY(cvk_init(device));
        const int kk = std::max(1, c.copy_group);
        nslots = std::max(c.pinned_slots, (2 * ((c.verify_batch + kk - 1) / kk) + c.fetch_threads + 2) * kk);
        nslots = (nslots + kk - 1) / kk * kk;
        copy_ev.resize(nslots), free_ev.resize(nslots);
        for (int i = 0; i < nslots; i++) {
            CU_TRY(cudaEventCreateWithFlags(&copy_ev[i], cudaEventDisableTiming));
            CU_TRY(cudaEventCreateWithFlags(&free_ev[i], cudaEventDisableTiming));
        }
        copy_streams.resize(static_cast<size_t>(std::max(1, std::min(c.copy_streams, c.fetch_threads))));
        for (auto& s : copy_streams) CU_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        CU_TRY(cudaStreamCreateWithFlags(&vstream, cudaStreamNonBlocking));
        CU_TRY(cudaEventCreateWithFlags(&done_ev, cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&entry_ev, cudaEventDisableTiming));
        reg.capacity = c.zero_copy ? static_cast<size_t>(std::max<int64_t>(c.register_cache, 0)) : 0;
        reg.min_age_sec = static_cast<double>(std::max<int64_t>(c.register_min_age_ms, 0)) / 1000.0;
        register_inline = c.register_threads <= 0 || reg.capacity == 0;
        // CPUs of the GPU's NUMA node: pinned pages and fetch threads stay next to the PCIe root
        int node = c.numa_node;  // -1: the GPU's node (auto); -2: do not bind the fetch threads
        if (node == -1) {
            char bus[64] = {0};
            if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) == cudaSuccess) {
                for (char* p = bus; *p; p++) *p = static_cast<char>(tolower(*p));
                std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/numa_node");
                if (f) f >> node;
            }
        }
        if (node >= 0) {
            std::ifstream f("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
            std::string s;
            if (f && std::getline(f, s)) {
                size_t p = 0;
                while (p < s.size()) {
                    const size_t c2 = s.find(',', p);
                    const std::string r = s.substr(p, c2 == std::string::npos ? std::string::npos : c2 - p);
                    const size_t d = r.find('-');
                    const int a = atoi(r.c_str()), b = d == std::string::npos ? a : atoi(r.c_str() + d + 1);
                    for (int x = a; x <= b; x++) cpus.push_back(x);
                    if (c2 == std::string::npos) break;
                    p = c2 + 1;
                }
            }
        }
        if (c.zero_copy && !register_inline) registrar.start(c.register_threads, device, &reg, cpus, c.register_when_idle ? &reads_in_flight : nullptr);
        if (c.zero_copy && c.arena) arena.start(std::max(1, c.register_threads), device, cpus, static_cast<size_t>(std::max<int64_t>(c.arena_register_slice, 0)));
        else arena.unsupported.store(true);
        return Err::ok();
    }

    void bind_thread() const {
        if (cpus.empty()) return;
        cpu_set_t set;
        CPU_ZERO(&set);
        for (int c : cpus) CPU_SET(c, &set);
        sched_setaffinity(0, sizeof(set), &set);
    }

    Err ensure(size_t need_slot_bytes, bool framed) {
        need_slot_bytes = (need_slot_bytes + 4095) & ~size_t(4095);
        if (need_slot_bytes > slot_bytes) {
            CU_TRY(cudaDeviceSynchronize());
            if (pinned) cudaFreeHost(pinned);
            if (d_stage) cudaFree(d_stage);
            pinned = nullptr, d_stage = nullptr, d_stage_bytes = 0;
            slot_bytes = need_slot_bytes;
            // allocate the ring from a thread bound to the GPU's node (the driver allocates and pins the pages in that
            // thread's context, so they land on its node; no extra first-touch pass)
            Err err;
            const double t0 = now_sec();
            std::thread t([&] {
                bind_thread();
                cudaSetDevice(device);
                cudaError_t e = cudaHostAlloc(&pinned, slot_bytes * nslots, cudaHostAllocDefault);
                if (e != cudaSuccess) err = Err::io(str_printf("cudaHostAlloc(%zu): %s", slot_bytes * nslots, cudaGetErrorString(e)));
            });
            t.join();
            ring_alloc_sec += now_sec() - t0;
            if (err) return err;
        }
        if (framed && d_stage_bytes < slot_bytes * nslots) {
            if (d_stage) cudaFree(d_stage);
            d_stage_bytes = slot_bytes * nslots;
            CU_TRY(cudaMalloc(&d_stage, d_stage_bytes));
        }
        return Err::ok();
    }

    ~GpuIngest() {
        registrar.stop();
        cudaSetDevice(device);
        cudaDeviceSynchronize();
        arena.stop();
        reg.clear();
        if (pinned) cudaFreeHost(pinned);
        if (d_stage) cudaFree(d_stage);
        if (d_tables) cudaFree(d_tables);
        if (h_result) cudaFreeHost(h_result);
        if (h_tables) cudaFreeHost(h_tables);
        for (auto e : copy_ev) cudaEventDestroy(e);
        for (auto e : free_ev) cudaEventDestroy(e);
        for (auto s : copy_streams) cudaStreamDestroy(s);
        if (vstream) cudaStreamDestroy(vstream);
        if (done_ev) cudaEventDestroy(done_ev);
        if (entry_ev) cudaEventDestroy(entry_ev);
    }
};

static std::mutex g_ing_mu;
static std::map<FsContext*, GpuIngest*> g_ingests;

GpuIngest* gpu_ingest_get(FsContext* ctx, Err* err) {
    std::lock_guard<std::mutex> lk(g_ing_mu);
    auto it = g_ingests.find(ctx);
    if (it != g_ingests.end()) return it->second;
    GpuIngest* g = new GpuIngest();
    *err = g->init(ctx->conf.b200);
    if (*err) {
        delete g;
        return nullptr;
    }
    g_ingests[ctx] = g;
    // the arenas named in the configuration are mapped + pinned from now on, in the background, off any read path
    if (ctx->conf.b200.zero_copy && ctx->conf.b200.arena)
        for (const std::string& spec : ctx->conf.b200.arena_dirs) {
            StorageDir d;
            if (parse_data_dir(spec, &d)) continue;
            g->arena.preregister_dir((ctx->conf.cluster_id.empty() ? d.path : d.path + "/" + ctx->conf.cluster_id) + "/arena");
        }
    return g;
}

Err gpu_ingest_preregister(FsContext* ctx) {
    Err e;
    gpu_ingest_get(ctx, &e);
    return e;
}

void gpu_ingest_arena_stats(FsContext* ctx, uint64_t out[5]) {
    memset(out, 0, 5 * sizeof(uint64_t));
    std::lock_guard<std::mutex> lk(g_ing_mu);
    auto it = g_ingests.find(ctx);
    if (it == g_ingests.end()) return;
    double sec = 0;
    it->second->arena.stats(&out[0], &out[1], &sec);
    out[2] = static_cast<uint64_t>(sec * 1e6), out[3] = it->second->arena.dma_jobs.load(), out[4] = it->second->arena.dma_bytes.load();
}

void gpu_ingest_wait_registered(FsContext* ctx) {
    GpuIngest* g = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_ing_mu);
        auto it = g_ingests.find(ctx);
        if (it != g_ingests.end()) g = it->second;
    }
    if (g) g->registrar.drain(), g->arena.drain();
}

void gpu_ingest_release(FsContext* ctx) {
    std::lock_guard<std::mutex> lk(g_ing_mu);
    auto it = g_ingests.find(ctx);
    if (it == g_ingests.end()) return;
    delete it->second;
    g_ingests.erase(it);
}

// ------------------------------------------------------------------ GpuFsReader

Err GpuFsReader::open(FsContext* ctx, const std::string& path, std::unique_ptr<GpuFsReader>* out) {
    std::unique_ptr<GpuFsReader> r(new GpuFsReader());
    r->ctx_ = ctx;
    CV_RETURN_IF_ERR(ctx->ns.get_block_locations(path, &r->fbp_));
    Err e;
    r->ing_ = gpu_ingest_get(ctx, &e);
    if (e) return e;
    *out = std::move(r);
    return Err::ok();
}

GpuFsReader::~GpuFsReader() {
    if (ing_) {
        std::lock_guard<std::mutex> lk(ing_->mu);
        harvest();
        if (ing_->pending_owner == this) ing_->pending_owner = nullptr;
    }
}

Err GpuFsReader::seek(int64_t pos) {
    if (pos < 0) return Err::common("Cannot seek to negative offset");
    // past-EOF positions are legal through FsReader (FsReaderParallel::seek clamps, fs_reader_parallel.rs:175-181): reads return 0
    pos_ = pos;
    return Err::ok();
}

Err GpuFsReader::complete() {
    uint64_t s, v;
    uint32_t b;
    return verify(&s, &b, &v);
}

Err GpuFsReader::fuse_read_device(int64_t want, void* d_scratch, void* d_page_base, const uint64_t* page_offsets, int64_t n_pages, int64_t page_size,
                                   void* stream, int64_t* n) {
    *n = 0;
    if (page_size <= 0) return Err::common("page_size must be positive");
    const int64_t take = std::max<int64_t>(0, std::min(want, len() - pos_));
    const int64_t need_pages = (take + page_size - 1) / page_size;
    if (need_pages > n_pages) return Err::common("not enough page buffers for the reply");
    PageScatter ps;
    ps.d_page_base = static_cast<uint8_t*>(d_page_base), ps.page_offsets = page_offsets, ps.n_pages = need_pages, ps.page_size = page_size, ps.total = take;
    return read_device_impl(d_scratch, take, stream, n, need_pages > 0 ? &ps : nullptr);
}

Err GpuFsReader::read_device(void* d_dst, int64_t cap, void* stream, int64_t* n) { return read_device_impl(d_dst, cap, stream, n, nullptr); }

Err GpuFsReader::read_device_impl(void* d_dst, int64_t cap, void* stream, int64_t* n, const PageScatter* pages) {
    *n = 0;
    const int64_t end = std::min(len(), pos_ + std::max<int64_t>(cap, 0));
    if (end <= pos_) return Err::ok();
    std::vector<Job> jobs;
    int64_t p = pos_;
    while (p < end) {
        int64_t boff;
        size_t idx;
        CV_RETURN_IF_ERR((*fbp_).get_read_block(p, &boff, &idx));
        const int64_t blen = (*fbp_).block_locs[idx].block.len;
        const int64_t take = std::min(end - p, blen - boff);
        jobs.push_back(Job{&(*fbp_).block_locs[idx], boff, take, p - pos_, boff == 0 && take == blen});
        p += take;
    }
    CV_RETURN_IF_ERR(run_jobs(jobs, static_cast<uint8_t*>(d_dst), stream, pages));
    *n = end - pos_;
    pos_ = end;
    return Err::ok();
}

Err plan_shard(const FileBlocks& fb, int rank, int world, int64_t cap, std::vector<ShardJob>* out, int64_t* total) {
    out->clear();
    *total = 0;
    if (world <= 0 || rank < 0 || rank >= world) return Err::common("bad shard spec");
    const int64_t bs = fb.status.block_size;
    for (size_t b = static_cast<size_t>(rank), j = 0; b < fb.block_locs.size(); b += static_cast<size_t>(world), j++) {
        const int64_t blen = fb.block_locs[b].block.len;
        if (cap >= 0 && static_cast<int64_t>(j) * bs + blen > cap) return Err::common("destination too small for this shard");
        out->push_back(ShardJob{b, fb.starts[b], blen, static_cast<int64_t>(j) * bs});
        *total += blen;
    }
    return Err::ok();
}

Err GpuFsReader::read_device_sharded(int rank, int world, void* d_dst, int64_t cap, void* stream, int64_t* n) {
    *n = 0;
    std::vector<ShardJob> plan;
    int64_t total = 0;
    CV_RETURN_IF_ERR(plan_shard(*fbp_, rank, world, cap, &plan, &total));
    std::vector<Job> jobs;
    for (const auto& p : plan) jobs.push_back(Job{&(*fbp_).block_locs[p.block], 0, p.len, p.dst_off, true});
    CV_RETURN_IF_ERR(run_jobs(jobs, static_cast<uint8_t*>(d_dst), stream));
    *n = total;
    return Err::ok();
}

namespace {

// Wait for `cond()`: a short spin, then sleep in growing steps so waiting threads do not starve the worker threads.
template <typename F>
static inline void backoff_wait(F cond) {
    for (int i = 0; i < 64; i++) {
        if (cond()) return;
        std::this_thread::yield();
    }
    unsigned us = 10;
    while (!cond()) {
        usleep(us);
        if (us < 200) us *= 2;
    }
}

}  // namespace

enum FetchMode { kFetchShortCircuit = 0, kFetchFramedVerbatim = 1 };

// Fetch one job's bytes into `slot`.
//   short-circuit    payload only (pread of the block file the worker named)
//   framed verbatim  the response stream exactly as received: 22-byte prefixes + payloads (unpacked on the GPU by K2, which
//                    also clips the last chunk of a range that stops short of the block end)
static Err fetch_job(FsContext* ctx, const LocatedBlock& lb, int64_t block_off, int64_t n, FetchMode mode, int64_t chunk, uint8_t* slot,
                     std::unique_ptr<BlockClient>* conn, int64_t* req_id_out, size_t* wire_bytes) {
    Err last = ctx->no_available_worker(lb.locs);
    for (const WorkerAddress& loc : lb.locs) {
        if (!*conn || !((*conn)->addr() == loc) || (*conn)->broken) {
            if (*conn) ctx->release(std::move(*conn));
            last = ctx->acquire_read(loc, conn);
            if (last) continue;
        }
        BlockClient* c = conn->get();
        const int64_t req_id = new_req_id();
        *req_id_out = req_id;
        BlockReadResponse resp;
        if (mode == kFetchFramedVerbatim) {
            // Open + every Running request + Complete in one write (the worker serves them in order, read_handler.rs:60-207).  The
            // worker answers each Running with min(chunk, block_len - pos) bytes, so the last frame of a range that stops short of
            // the block end carries bytes past it: they are received like the rest and clipped by K2 (CvStreamDesc.tail_clip).
            const int64_t nfr = (n + chunk - 1) / chunk;
            n = std::min<int64_t>(nfr * chunk, lb.block.len - block_off);  // payload bytes on the wire
            last = c->send_block_read_pipeline(ctx->conf.client, lb.block, block_off, req_id, chunk, nfr, &resp);
            if (last) continue;
            uint8_t* w = slot;
            int64_t left = n;
            for (int64_t f = 0; f < nfr && !last; f++) {
                last = recv_exact(c->fd(), w, kProtocolSize);
                Protocol p;
                if (!last) last = decode_protocol(w, &p);
                if (last) break;
                const int64_t want = std::min(chunk, left);
                if (!p.is_success() || p.header_len != 0 || p.data_len != want) {
                    // error response (or an unexpected chunk): drain this frame, report it, drop the connection
                    std::string body(static_cast<size_t>(p.header_len + p.data_len), '\0');
                    if (!body.empty() && recv_exact(c->fd(), &body[0], body.size())) c->broken = true;
                    last = p.is_success() ? Err::common(str_printf("unexpected chunk length %d, expected %lld", p.data_len, (long long)want))
                                          : decode_error_body(reinterpret_cast<const uint8_t*>(body.data()) + p.header_len, static_cast<size_t>(p.data_len));
                    break;
                }
                last = recv_exact(c->fd(), w + kProtocolSize, static_cast<size_t>(want));
                w += kProtocolSize + want, left -= want;
            }
            if (last) {
                c->broken = true;  // responses of the remaining pipelined requests may still be in flight
                continue;
            }
            *wire_bytes = static_cast<size_t>(w - slot);
            return Err::ok();  // the Complete went out with the rest; its answer is consumed in front of this connection's next request
        }
        const int64_t open_chunk = ctx->read_chunk_size();
        last = c->open_block(ctx->conf.client, lb.block, block_off, lb.block.len, req_id, 0, true, open_chunk, &resp, ctx->conf.b200.arena);
        if (last) continue;
        int32_t seq = 0;
        const int64_t base_off = resp.has_arena ? resp.arena_off : 0;  // arena block: an extent inside the segment file
        if (mode == kFetchShortCircuit) {
            if (!resp.has_path) {
                last = Err::common("read_context.path is none");
                continue;
            }
            const int fd = ::open(resp.path.c_str(), O_RDONLY | O_CLOEXEC);
            if (fd < 0) {
                last = Err::io(str_printf("open %s: %s", resp.path.c_str(), strerror(errno)));
                continue;
            }
            int64_t got = 0;
            while (got < n) {
                const ssize_t r = pread(fd, slot + got, static_cast<size_t>(n - got), base_off + block_off + got);
                if (r < 0 && errno == EINTR) continue;
                if (r <= 0) {
                    last = Err::io(str_printf("read block file: %s", r == 0 ? "unexpected eof" : strerror(errno)));
                    break;
                }
                got += r;
            }
            ::close(fd);
            if (got < n) continue;
            *wire_bytes = static_cast<size_t>(n);
        }
        last = c->read_commit_deferred(lb.block, req_id, seq + 1);  // its answer is consumed in front of this connection's next request
        if (last) continue;
        return Err::ok();
    }
    return last;
}

// Open(short_circuit=true) on the first replica that answers; returns the block file path.
static Err open_short_circuit(FsContext* ctx, const LocatedBlock& lb, int64_t block_off, std::unique_ptr<BlockClient>* conn, int64_t* req_id,
                              BlockReadResponse* out) {
    Err last = ctx->no_available_worker(lb.locs);
    for (const WorkerAddress& loc : lb.locs) {
        if (!*conn || !((*conn)->addr() == loc) || (*conn)->broken) {
            if (*conn) ctx->release(std::move(*conn));
            last = ctx->acquire_read(loc, conn);
            if (last) continue;
        }
        *req_id = new_req_id();
        BlockReadResponse resp;
        last = (*conn)->open_block(ctx->conf.client, lb.block, block_off, lb.block.len, *req_id, 0, true, ctx->read_chunk_size(), &resp, ctx->conf.b200.arena);
        if (last) continue;
        if (!resp.has_path) {
            last = Err::common("read_context.path is none");
            continue;
        }
        *out = resp;
        return Err::ok();
    }
    return last;
}

// Pull the last call's per-block CRCs / mismatch count / frame flags (already copied to the pinned mirror on vstream).
Err GpuFsReader::harvest() {
    if (!pending_.active) return Err::ok();
    GpuIngest& G = *ing_;
    cudaSetDevice(G.device);
    CU_TRY(cudaStreamSynchronize(G.vstream));
    const uint32_t* crc = reinterpret_cast<const uint32_t*>(G.h_result);
    const size_t J = pending_.jobs;
    for (size_t j = pending_.f0; j < pending_.f1; j++) sum_crc_ += crc[j];
    n_verified_ += pending_.n_compared;
    stats_.verified += pending_.n_compared;
    n_bad_ += crc[J];  // mismatch counter written by cvk_verify_crcs
    const uint32_t* ferr = crc + J + 4;
    for (size_t f = 0; f < pending_.frames; f++)
        if (ferr[f]) {
            n_bad_frames_++;
            if (!first_frame_err_) first_frame_err_ = ferr[f];
        }
    pending_.active = false;
    held_maps_.clear();  // every copy that read from these mappings has completed (vstream waited on them)
    if (G.pending_owner == this) G.pending_owner = nullptr;
    if (n_bad_frames_) return Err(kAbnormalData, str_printf("%llu frame prefixes failed validation (first flags 0x%x)", (unsigned long long)n_bad_frames_, first_frame_err_));
    return Err::ok();
}

Err GpuFsReader::verify(uint64_t* sum_crc, uint32_t* n_bad, uint64_t* n_verified) {
    Err e;
    if (ing_) {
        std::lock_guard<std::mutex> lk(ing_->mu);
        e = harvest();
    }
    *sum_crc = sum_crc_, *n_bad = n_bad_, *n_verified = n_verified_;
    return e;
}

Err GpuFsReader::run_jobs(const std::vector<Job>& jobs, uint8_t* d_dst, void* user_stream, const PageScatter* pages) {
    const size_t J = jobs.size();
    if (J == 0) return Err::ok();
    const double t_start = now_sec();
    GpuIngest& G = *ing_;
    struct InFlight {
        std::atomic<int>& n;
        explicit InFlight(std::atomic<int>& c) : n(c) { n.fetch_add(1, std::memory_order_acq_rel); }
        ~InFlight() { n.fetch_sub(1, std::memory_order_acq_rel); }
    } in_flight(G.reads_in_flight);
    std::lock_guard<std::mutex> call_lock(G.mu);
    CU_TRY(cudaSetDevice(G.device));
    {
        cudaPointerAttributes pa;
        if (cudaPointerGetAttributes(&pa, d_dst) != cudaSuccess || pa.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            return Err::common("cv_read_device: destination is not device memory");
        }
        if (pa.device != G.device)
            return Err::common(str_printf("cv_read_device: destination lives on device %d but [b200] device = %d", pa.device, G.device));
    }
    if (G.pending_owner && G.pending_owner != this) CV_RETURN_IF_ERR(G.pending_owner->harvest());  // shared tables
    CV_RETURN_IF_ERR(harvest());
    // everything this call writes into d_dst is ordered after what the caller's stream had queued at entry (a buffer fresh from
    // a stream-ordered allocator, kernels still reading it): the copy streams and the verify stream wait for that point
    CU_TRY(cudaEventRecord(G.entry_ev, static_cast<cudaStream_t>(user_stream)));
    for (auto cs : G.copy_streams) CU_TRY(cudaStreamWaitEvent(cs, G.entry_ev, 0));
    CU_TRY(cudaStreamWaitEvent(G.vstream, G.entry_ev, 0));
    const B200Conf& bc = ctx_->conf.b200;
    const ClientConf& cc = ctx_->conf.client;
    const int poly = bc.verify_poly ? 1 : 0;
    const int64_t chunk = std::min<int64_t>(std::max<int64_t>(bc.gpu_chunk_size, 4096), kMaxDataSize);

    // ---- per-job mode.  Short-circuit (the reference default for a same-host worker, client_conf.rs:339) only when
    // every block of this call has a local replica; otherwise the whole call runs framed (any worker serves those).
    enum : uint8_t { kPlain = 0, kFramed = 1, kHole = 3 };
    std::vector<uint8_t> mode(J, kPlain);
    bool call_framed = false;
    for (size_t j = 0; j < J; j++) {
        const LocatedBlock& lb = (*jobs[j].lb);
        if (lb.locs.empty()) {
            if (!lb.block.has_alloc_opts) return ctx_->no_available_worker(lb.locs);
            mode[j] = kHole;
            continue;
        }
        bool local = false;
        for (const auto& a : lb.locs) local |= ctx_->is_local_worker(a);
        if (!(cc.short_circuit && local)) call_framed = true;
    }
    size_t need_slot = 0, F = 0;
    std::vector<uint32_t> first_frame(J + 1, 0);
    bool any_verbatim = false;
    std::vector<int64_t> wire_payload(J, 0);  // framed jobs: payload bytes the worker sends (>= n when the range stops short of the block end)
    for (size_t j = 0; j < J; j++) {
        first_frame[j] = static_cast<uint32_t>(F);
        size_t bytes = static_cast<size_t>(jobs[j].n);
        if (mode[j] != kHole && call_framed) {
            // every framed job is received verbatim and unpacked by K2; a range that stops short of its block's end gets the
            // worker's whole last chunk and K2 clips it (CvStreamDesc.tail_clip) -- no host-side unpacking anywhere
            mode[j] = kFramed;
            const int64_t nfr = (jobs[j].n + chunk - 1) / chunk;
            wire_payload[j] = std::min<int64_t>(nfr * chunk, (*jobs[j].lb).block.len - jobs[j].block_off);
            bytes = static_cast<size_t>(wire_payload[j] + nfr * kProtocolSize);
            F += static_cast<size_t>(nfr);
            any_verbatim = true;
        }
        need_slot = std::max(need_slot, bytes);
    }
    first_frame[J] = static_cast<uint32_t>(F);
    // the pinned ring (and the device staging ring for verbatim frames) is only materialised when a group needs it:
    // the zero-copy path never touches it
    std::once_flag ring_once;
    Err ring_err;
    auto ensure_ring = [&]() -> Err {
        std::call_once(ring_once, [&] { ring_err = G.ensure(need_slot, any_verbatim); });
        return ring_err;
    };
    if (!(bc.zero_copy && !call_framed)) CV_RETURN_IF_ERR(ensure_ring());

    // ---- copy groups: k consecutive jobs share one super-slot and, when they are contiguous, one cudaMemcpyAsync
    const size_t k = static_cast<size_t>(std::max(1, std::min(bc.copy_group, G.nslots / 4)));
    const size_t NG = (J + k - 1) / k;                    // copy groups in this call
    const size_t NS = static_cast<size_t>(G.nslots) / k;  // super-slots in the ring
    const size_t vgroups = std::max<size_t>(1, (static_cast<size_t>(std::max(1, bc.verify_batch)) + k - 1) / k);  // copy groups per verify launch
    const size_t B = vgroups * k;

    // ---- device tables (shared by all readers of this context): off[J] len[J] | expect[J] crc[J] nbad[4] ferr[F] | streams[J] fdesc[F]
    auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t o_off = 0, o_len = up(o_off + 8 * J), o_exp = up(o_len + 8 * J), o_skip = up(o_exp + 4 * J), o_crc = up(o_skip + J);
    const size_t res_words = J + 4 + F;
    const size_t o_streams = up(o_crc + 4 * res_words), o_fdesc = up(o_streams + sizeof(CvStreamDesc) * J);
    const size_t n_segs = pages ? static_cast<size_t>(pages->n_pages) : 0;
    const size_t o_segs = up(o_fdesc + sizeof(CvFrameDesc) * F);
    const size_t tables_bytes = up(o_segs + sizeof(CvSeg) * n_segs);
    CV_RETURN_IF_ERR(G.ensure_tables(tables_bytes, 4 * res_words));
    uint8_t* T = G.d_tables;
    // host image of off/len/expect/skip (+ the stream descriptors): pinned, owned by the context, rewritten only after the
    // previous call's results were harvested (its uploads have long executed by then)
    uint8_t* h = G.h_tables;
    uint64_t* h_off = reinterpret_cast<uint64_t*>(&h[o_off]);
    uint64_t* h_len = reinterpret_cast<uint64_t*>(&h[o_len]);
    uint32_t* h_exp = reinterpret_cast<uint32_t*>(&h[o_exp]);
    uint8_t* h_skip = &h[o_skip];
    size_t f0 = J, f1 = 0, n_compared = 0;
    for (size_t j = 0; j < J; j++) {
        const LocatedBlock& lb = (*jobs[j].lb);
        h_off[j] = static_cast<uint64_t>(jobs[j].dst_off);
        h_len[j] = static_cast<uint64_t>(jobs[j].n);
        h_exp[j] = poly ? lb.crc32c : lb.crc32;
        h_skip[j] = !(jobs[j].full && lb.has_crc && mode[j] != kHole);
        if (!h_skip[j]) {
            f0 = std::min(f0, j), f1 = std::max(f1, j + 1);
            n_compared++;
        }
    }
    if (f0 >= f1) f0 = f1 = 0;
    // every whole block the manifest holds a CRC for is compared; holes, partial ranges and blocks without a manifest CRC are
    // masked out one by one (their CRCs are still computed, and summed when they lie inside [f0,f1))
    const bool compare = bc.verify && n_compared > 0;
    CU_TRY(cudaMemcpyAsync(T, h, o_crc, cudaMemcpyHostToDevice, G.vstream));
    if (n_segs) {  // the page scatter's segment table rides in the same pinned image
        CvSeg* hs = reinterpret_cast<CvSeg*>(h + o_segs);
        for (size_t i = 0; i < n_segs; i++) {
            hs[i].src_off = static_cast<uint64_t>(i) * static_cast<uint64_t>(pages->page_size), hs[i].dst_off = pages->page_offsets[i];
            hs[i].len = static_cast<uint64_t>(std::min<int64_t>(pages->page_size, pages->total - static_cast<int64_t>(i) * pages->page_size));
        }
        CU_TRY(cudaMemcpyAsync(T + o_segs, hs, sizeof(CvSeg) * n_segs, cudaMemcpyHostToDevice, G.vstream));
    }
    CU_TRY(cudaMemsetAsync(T + o_crc, 0, 4 * res_words, G.vstream));
    CvStreamDesc* sd = reinterpret_cast<CvStreamDesc*>(h + o_streams);
    if (any_verbatim) {
        for (size_t j = 0; j < J; j++) {
            CvStreamDesc& d = sd[j];
            memset(&d, 0, sizeof(d));
            const size_t ss = (j / k) % NS;
            d.wire_off = (ss * k + j % k) * G.slot_bytes, d.dst_off = h_off[j], d.block_len = mode[j] == kFramed ? static_cast<uint64_t>(wire_payload[j]) : 0;
            d.tail_clip = mode[j] == kFramed ? static_cast<uint32_t>(wire_payload[j] - jobs[j].n) : 0;
            d.chunk_size = static_cast<uint32_t>(chunk), d.first_seq_id = 1, d.block = static_cast<uint32_t>(j % B);
            d.first_frame = first_frame[j], d.code = kCodeReadBlock, d.status = 0x03;
        }
    }

    // ---- fetch threads
    struct Shared {
        std::atomic<size_t> next_group{0};
        std::atomic<bool> abort{false};
        std::mutex err_mu;
        Err err;
        void fail(const Err& e) {
            std::lock_guard<std::mutex> lk(err_mu);
            if (!err) err = e;
            abort.store(true);
        }
    } st;
    std::vector<std::atomic<int>> copied(NG);
    std::vector<std::atomic<int64_t>> released(NS);  // per super-slot: last copy group whose release event is recorded
    for (auto& c : copied) c.store(0);
    for (auto& r : released) r.store(-1);
    std::vector<uint8_t> group_verbatim(NG, 0);
    for (size_t g = 0; g < NG; g++)
        for (size_t j = g * k; j < std::min(J, g * k + k); j++) group_verbatim[g] |= mode[j] == kFramed;
    std::vector<int64_t> req_ids(J, 0);
    std::atomic<bool> use_mapped{bc.zero_copy};
    std::atomic<bool> use_gds{!call_framed && bc.gds && gds_info().available};
    std::atomic<uint64_t> gds_bytes{0};
    std::mutex held_mu;
    const int T_threads = static_cast<int>(std::min<size_t>(static_cast<size_t>(std::max(1, bc.fetch_threads)), NG));
    std::vector<double> fetch_sec(static_cast<size_t>(T_threads), 0.0);
    std::vector<uint64_t> h2d(static_cast<size_t>(T_threads), 0);
    auto worker = [&](int t, bool own_thread) {
        if (own_thread) G.bind_thread();  // an inline call (single copy group: small reads) must not re-pin the caller
        cudaSetDevice(G.device);
        cudaStream_t cs = G.copy_streams[static_cast<size_t>(t) % G.copy_streams.size()];
        std::unique_ptr<BlockClient> conn;
        for (;;) {
            const size_t g = st.next_group.fetch_add(1);
            if (g >= NG || st.abort.load()) break;
            const size_t ss = g % NS, j0 = g * k, j1 = std::min(J, j0 + k);
            if (g >= NS) {  // wait until the super-slot's previous tenant has been released, then for its event
                const int64_t want = static_cast<int64_t>(g - NS);
                backoff_wait([&] { return released[ss].load(std::memory_order_acquire) >= want || st.abort.load(); });
                if (st.abort.load()) break;
                cudaEventSynchronize(group_verbatim[g - NS] ? G.free_ev[ss] : G.copy_ev[ss]);
            }
            bool all_plain = true;
            for (size_t j = j0; j < j1; j++) all_plain = all_plain && mode[j] == kPlain;
            // ---- GPUDirect Storage: blocks of a disk tier go file -> HBM by cuFileRead, no host ring
            bool all_disk = all_plain && use_gds.load(std::memory_order_relaxed);
            for (size_t j = j0; j < j1 && all_disk; j++) all_disk = (*jobs[j].lb).block.storage_type != kStorageMem;
            if (all_disk) {
                const double t0 = now_sec();
                Err e;
                backoff_wait([&] { return cudaEventQuery(G.entry_ev) != cudaErrorNotReady; });  // cuFile knows nothing of the caller's stream
                for (size_t j = j0; j < j1 && !e; j++) {
                    BlockReadResponse resp;
                    int64_t rid = 0;
                    e = open_short_circuit(ctx_, (*jobs[j].lb), jobs[j].block_off, &conn, &rid, &resp);
                    if (!e) e = gds_read(resp.path, d_dst + jobs[j].dst_off, jobs[j].n, (resp.has_arena ? resp.arena_off : 0) + jobs[j].block_off);
                    if (!e) e = conn->read_commit_deferred((*jobs[j].lb).block, rid, 1);
                    if (!e) gds_bytes += static_cast<uint64_t>(jobs[j].n);
                }
                fetch_sec[static_cast<size_t>(t)] += now_sec() - t0;
                if (e && e.kind == kUnsupported) {
                    use_gds.store(false);  // this file system / this box cannot do it: the pinned ring takes over (the group is redone below)
                } else {
                    cudaError_t ce = e ? cudaSuccess : cudaEventRecord(G.copy_ev[ss], cs);
                    if (e || ce != cudaSuccess) {
                        st.fail(e ? e : Err::io(str_printf("event record: %s", cudaGetErrorString(ce))));
                        break;
                    }
                    released[ss].store(static_cast<int64_t>(g), std::memory_order_release);
                    copied[g].store(1, std::memory_order_release);
                    continue;
                }
            }
            // ---- zero-copy: DMA out of registered mmaps of the block files (mem tier), no pinned-slot copy
            if (all_plain && use_mapped.load(std::memory_order_relaxed)) {
                const double t0 = now_sec();
                std::vector<std::string> paths(j1 - j0);
                std::vector<int64_t> lens(j1 - j0), rids(j1 - j0), base_offs(j1 - j0, 0);
                Err e;
                size_t n_arena = 0;
                for (size_t j = j0; j < j1 && !e; j++) {
                    const LocatedBlock& lb = (*jobs[j].lb);
                    BlockReadResponse resp;
                    e = open_short_circuit(ctx_, lb, jobs[j].block_off, &conn, &rids[j - j0], &resp);
                    paths[j - j0] = resp.path, lens[j - j0] = lb.block.len;
                    if (resp.has_arena) base_offs[j - j0] = resp.arena_off, n_arena++;
                }
                // ---- mem arena: every block of the group is an extent of a segment this context pinned once
                if (!e && n_arena == j1 - j0 && !G.arena.unsupported.load(std::memory_order_relaxed)) {
                    std::vector<std::shared_ptr<ArenaSeg>> segs(j1 - j0);
                    for (size_t j = j0; j < j1 && !e; j++) {
                        if (j > j0 && paths[j - j0] == paths[j - j0 - 1]) segs[j - j0] = segs[j - j0 - 1];
                        else e = G.arena.get(paths[j - j0], &segs[j - j0]);
                        if (!e && static_cast<size_t>(base_offs[j - j0] + jobs[j].block_off + jobs[j].n) > segs[j - j0]->bytes) e = Err::io("arena extent lies outside its segment");
                    }
                    if (!e) {
                        cudaError_t ce = cudaSuccess;
                        // one cudaMemcpyAsync per run of jobs that are back to back in the segment AND in the destination
                        for (size_t j = j0; j < j1 && ce == cudaSuccess;) {
                            const uint8_t* src = segs[j - j0]->base + base_offs[j - j0] + jobs[j].block_off;
                            size_t len = static_cast<size_t>(jobs[j].n), r = j + 1;
                            while (r < j1 && segs[r - j0] == segs[j - j0] && segs[r - j0]->base + base_offs[r - j0] + jobs[r].block_off == src + len &&
                                   jobs[r].dst_off == jobs[j].dst_off + static_cast<int64_t>(len))
                                len += static_cast<size_t>(jobs[r].n), r++;
                            // a copy never spans two separately registered slices of the segment
                            const ArenaSeg& sg = *segs[j - j0];
                            for (size_t done = 0; done < len && ce == cudaSuccess;) {
                                const size_t in_seg = static_cast<size_t>(src - sg.base) + done;
                                const size_t piece = std::min(len - done, (in_seg / sg.slice + 1) * sg.slice - in_seg);
                                ce = cudaMemcpyAsync(d_dst + jobs[j].dst_off + done, src + done, piece, cudaMemcpyHostToDevice, cs);
                                done += piece;
                            }
                            h2d[static_cast<size_t>(t)] += len;
                            j = r;
                        }
                        if (ce == cudaSuccess) ce = cudaEventRecord(G.copy_ev[ss], cs);
                        for (size_t j = j0; j < j1 && !e; j++) e = conn->read_commit_deferred((*jobs[j].lb).block, rids[j - j0], 1);
                        fetch_sec[static_cast<size_t>(t)] += now_sec() - t0;
                        if (e || ce != cudaSuccess) {
                            st.fail(e ? e : Err::io(str_printf("H2D enqueue: %s", cudaGetErrorString(ce))));
                            break;
                        }
                        G.arena.dma_jobs += j1 - j0;
                        for (size_t j = j0; j < j1; j++) G.arena.dma_bytes += static_cast<uint64_t>(jobs[j].n);
                        released[ss].store(static_cast<int64_t>(g), std::memory_order_release);
                        copied[g].store(1, std::memory_order_release);
                        continue;
                    }
                    if (e.kind == kUnsupported) e = Err::ok();  // segments cannot be pinned here: the group goes through the ring below
                }
                std::shared_ptr<RegMapping> m;
                bool via_ring = n_arena > 0;  // arena extents (mixed group, or segments that cannot be pinned): pread out of the segment file
                if (!e && !via_ring) {
                    std::string key;
                    for (const auto& p : paths) key += p, key += '|';
                    std::vector<uint64_t> stamps;
                    if (stat_stamps(paths, &stamps)) m = G.reg.find(key, stamps);
                    if (!m) G.reg.misses++;
                    if (!m && G.registrar.unsupported.load()) e = Err(kUnsupported, "cudaHostRegister of file mappings is not supported here");
                    if (!m && !e) {
                        size_t group_bytes = 0;
                        for (int64_t l : lens) group_bytes += (static_cast<size_t>(l) + 4095) / 4096 * 4096;
                        if (G.reg.capacity > 0 && !G.reg.can_admit(group_bytes)) {
                            // the cache is full of mappings in use or used moments ago (a scan larger than the cache): registering
                            // this group would be paid for and thrown away -- it goes through the ring, now and next time
                            G.reg.rejected++;
                            via_ring = true;
                        } else if (G.register_inline) {
                            e = map_and_register(paths, lens, &m, &stamps);
                            if (!e) {
                                m->key = key;
                                G.reg.insert(m);
                            }
                        } else {  // cold group: register it in the background for the next pass, move it through the ring now
                            G.registrar.submit(Registrar::Job{key, paths, lens});
                            via_ring = true;
                        }
                    }
                }
                cudaError_t ce = cudaSuccess;
                if (!e && via_ring) {
                    e = ensure_ring();
                    uint8_t* hs = G.pinned + ss * k * G.slot_bytes;
                    bool contiguous = true;
                    for (size_t j = j0 + 1; j < j1; j++) contiguous = contiguous && jobs[j].dst_off == jobs[j - 1].dst_off + jobs[j - 1].n;
                    if (contiguous && static_cast<size_t>(jobs[j1 - 1].dst_off + jobs[j1 - 1].n - jobs[j0].dst_off) > k * G.slot_bytes) contiguous = false;
                    for (size_t j = j0; j < j1 && !e && ce == cudaSuccess; j++) {
                        const size_t in_slot = contiguous ? static_cast<size_t>(jobs[j].dst_off - jobs[j0].dst_off) : (j - j0) * G.slot_bytes;
                        const int fd = ::open(paths[j - j0].c_str(), O_RDONLY | O_CLOEXEC);
                        if (fd < 0) {
                            e = Err::io(str_printf("open %s: %s", paths[j - j0].c_str(), strerror(errno)));
                            break;
                        }
                        int64_t got = 0;
                        while (got < jobs[j].n) {
                            const ssize_t r = pread(fd, hs + in_slot + got, static_cast<size_t>(jobs[j].n - got), base_offs[j - j0] + jobs[j].block_off + got);
                            if (r < 0 && errno == EINTR) continue;
                            if (r <= 0) {
                                e = Err::io(str_printf("read block file: %s", r == 0 ? "unexpected eof" : strerror(errno)));
                                break;
                            }
                            got += r;
                        }
                        ::close(fd);
                        if (!e && !contiguous) {
                            ce = cudaMemcpyAsync(d_dst + jobs[j].dst_off, hs + in_slot, static_cast<size_t>(jobs[j].n), cudaMemcpyHostToDevice, cs);
                            h2d[static_cast<size_t>(t)] += static_cast<size_t>(jobs[j].n);
                        }
                    }
                    if (!e && contiguous && ce == cudaSuccess) {
                        const size_t extent = static_cast<size_t>(jobs[j1 - 1].dst_off + jobs[j1 - 1].n - jobs[j0].dst_off);
                        ce = cudaMemcpyAsync(d_dst + jobs[j0].dst_off, hs, extent, cudaMemcpyHostToDevice, cs);
                        h2d[static_cast<size_t>(t)] += extent;
                    }
                    if (!e && ce == cudaSuccess) ce = cudaEventRecord(G.copy_ev[ss], cs);
                    for (size_t j = j0; j < j1 && !e; j++) e = conn->read_commit((*jobs[j].lb).block, rids[j - j0], 1);
                } else if (!e) {
                    // one copy when the group is whole blocks landing back to back, else one per job
                    bool whole = true;
                    for (size_t j = j0; j < j1; j++) {
                        whole = whole && jobs[j].block_off == 0 && (j + 1 == j1 || jobs[j].n == lens[j - j0]);
                        if (j > j0) whole = whole && jobs[j].dst_off == jobs[j - 1].dst_off + jobs[j - 1].n;
                    }
                    if (whole) {
                        const size_t extent = static_cast<size_t>(jobs[j1 - 1].dst_off + jobs[j1 - 1].n - jobs[j0].dst_off);
                        ce = cudaMemcpyAsync(d_dst + jobs[j0].dst_off, m->base, extent, cudaMemcpyHostToDevice, cs);
                        h2d[static_cast<size_t>(t)] += extent;
                    } else {
                        size_t moff = 0;
                        for (size_t j = j0; j < j1 && ce == cudaSuccess; j++) {
                            ce = cudaMemcpyAsync(d_dst + jobs[j].dst_off, m->base + moff + jobs[j].block_off, static_cast<size_t>(jobs[j].n), cudaMemcpyHostToDevice, cs);
                            h2d[static_cast<size_t>(t)] += static_cast<size_t>(jobs[j].n);
                            moff += (static_cast<size_t>(lens[j - j0]) + 4095) / 4096 * 4096;
                        }
                    }
                    if (ce == cudaSuccess) ce = cudaEventRecord(G.copy_ev[ss], cs);
                    {
                        std::lock_guard<std::mutex> lk(held_mu);
                        held_maps_.push_back(m);
                    }
                    for (size_t j = j0; j < j1 && !e; j++) e = conn->read_commit((*jobs[j].lb).block, rids[j - j0], 1);
                }
                fetch_sec[static_cast<size_t>(t)] += now_sec() - t0;
                if (e && e.kind == kUnsupported) {
                    use_mapped.store(false);  // cannot register file mappings here: fall back to the pinned ring below
                } else {
                    if (e || ce != cudaSuccess) {
                        st.fail(e ? e : Err::io(str_printf("H2D enqueue: %s", cudaGetErrorString(ce))));
                        break;
                    }
                    released[ss].store(static_cast<int64_t>(g), std::memory_order_release);
                    copied[g].store(1, std::memory_order_release);
                    continue;
                }
            }
            if (Err re = ensure_ring()) {
                st.fail(re);
                break;
            }
            uint8_t* hs = G.pinned + ss * k * G.slot_bytes;
            uint8_t* ds = G.d_stage ? G.d_stage + ss * k * G.slot_bytes : nullptr;
            // plain jobs mirror the destination layout inside the super-slot so that one copy moves the whole group
            bool one_copy = !group_verbatim[g];
            for (size_t j = j0; j < j1 && one_copy; j++) {
                one_copy = mode[j] == kPlain;
                if (j > j0) one_copy = one_copy && jobs[j].dst_off == jobs[j - 1].dst_off + jobs[j - 1].n;
            }
            if (one_copy && static_cast<size_t>(jobs[j1 - 1].dst_off + jobs[j1 - 1].n - jobs[j0].dst_off) > k * G.slot_bytes) one_copy = false;
            cudaError_t ce = cudaSuccess;
            size_t wire_extent = 0;
            bool failed = false;
            for (size_t j = j0; j < j1 && !failed; j++) {
                const Job& job = jobs[j];
                if (mode[j] == kHole) {
                    ce = cudaMemsetAsync(d_dst + job.dst_off, 0, static_cast<size_t>(job.n), cs);  // block_reader_hole.rs:69-79
                    failed = ce != cudaSuccess;
                    continue;
                }
                const size_t in_slot = one_copy ? static_cast<size_t>(job.dst_off - jobs[j0].dst_off) : (j - j0) * G.slot_bytes;
                size_t wire = 0;
                const double t0 = now_sec();
                const FetchMode fm = mode[j] == kPlain ? kFetchShortCircuit : kFetchFramedVerbatim;
                Err e = fetch_job(ctx_, (*job.lb), job.block_off, job.n, fm, chunk, hs + in_slot, &conn, &req_ids[j], &wire);
                fetch_sec[static_cast<size_t>(t)] += now_sec() - t0;
                if (e) {
                    st.fail(e.ctx(str_printf("block %lld", (long long)(*job.lb).block.id)));
                    failed = true;
                    break;
                }
                if (group_verbatim[g]) {
                    if (mode[j] == kFramed) wire_extent = in_slot + wire;  // copied below in one piece
                    else ce = cudaMemcpyAsync(d_dst + job.dst_off, hs + in_slot, wire, cudaMemcpyHostToDevice, cs), h2d[static_cast<size_t>(t)] += wire;
                } else if (!one_copy) {
                    ce = cudaMemcpyAsync(d_dst + job.dst_off, hs + in_slot, wire, cudaMemcpyHostToDevice, cs), h2d[static_cast<size_t>(t)] += wire;
                }
                failed = ce != cudaSuccess;
            }
            if (st.abort.load() && failed && ce == cudaSuccess) break;
            if (!failed && group_verbatim[g] && wire_extent) {
                ce = cudaMemcpyAsync(ds, hs, wire_extent, cudaMemcpyHostToDevice, cs);
                h2d[static_cast<size_t>(t)] += wire_extent;
            } else if (!failed && one_copy) {
                const size_t extent = static_cast<size_t>(jobs[j1 - 1].dst_off + jobs[j1 - 1].n - jobs[j0].dst_off);
                ce = cudaMemcpyAsync(d_dst + jobs[j0].dst_off, hs, extent, cudaMemcpyHostToDevice, cs);
                h2d[static_cast<size_t>(t)] += extent;
            }
            if (ce == cudaSuccess && !failed) ce = cudaEventRecord(G.copy_ev[ss], cs);
            if (ce != cudaSuccess) {
                st.fail(Err::io(str_printf("H2D enqueue: %s", cudaGetErrorString(ce))));
                break;
            }
            if (failed) break;
            if (!group_verbatim[g]) released[ss].store(static_cast<int64_t>(g), std::memory_order_release);
            copied[g].store(1, std::memory_order_release);
        }
        if (conn) {
            // multi-group reads: settle the deferred Completes here (their answers are long in); a single-group read (the
            // latency path, C5) parks the connection with its last answer outstanding and the next request consumes it
            if (NG > 1) conn->drain_pending();
            ctx_->release(std::move(conn));
        }
    };
    std::vector<std::thread> threads;
    // A verbatim (framed) group's slot is only released by the verifier below, so a single fetch worker running inline on this
    // thread would wait for itself once the groups outnumber the ring's super-slots: it gets its own thread then.
    if (T_threads == 1 && (NG <= NS || !any_verbatim)) worker(0, false);  // small read (FUSE-shaped, C5): no thread spawn on the latency path
    else
        for (int t = 0; t < T_threads; t++) threads.emplace_back(worker, t, true);

    // ---- verifier: this thread walks the copy groups in order, `vgroups` at a time
    Err verr;
    const uint64_t launches0 = cvk_launch_count();
    const uint64_t* d_off = reinterpret_cast<const uint64_t*>(T + o_off);
    const uint64_t* d_len = reinterpret_cast<const uint64_t*>(T + o_len);
    uint32_t* d_crc = reinterpret_cast<uint32_t*>(T + o_crc);
    uint32_t* d_ferr = d_crc + J + 4;
    CvStreamDesc* d_streams = reinterpret_cast<CvStreamDesc*>(T + o_streams);
    CvFrameDesc* d_fdesc = reinterpret_cast<CvFrameDesc*>(T + o_fdesc);
    for (size_t v0 = 0; v0 < NG && !verr; v0 += vgroups) {
        const size_t v1 = std::min(NG, v0 + vgroups);
        for (size_t g = v0; g < v1; g++)
            backoff_wait([&] { return copied[g].load(std::memory_order_acquire) != 0 || st.abort.load(); });
        if (st.abort.load()) break;
        const size_t g0 = v0 * k, g1 = std::min(J, v1 * k);
        uint64_t gbytes = 0;
        bool gframed = false;
        for (size_t g = v0; g < v1; g++) {
            cudaStreamWaitEvent(G.vstream, G.copy_ev[g % NS], 0);
            gframed |= group_verbatim[g] != 0;
        }
        for (size_t j = g0; j < g1; j++) gbytes += h_len[j];
        if (!gframed && bc.verify) {  // K1 over the landed bytes
            int rc = cvk_crc_blocks(d_dst, d_off + g0, d_len + g0, static_cast<uint32_t>(g1 - g0), poly, gbytes, d_crc + g0, G.vstream);
            if (rc) verr = Err::io(str_printf("cvk_crc_blocks: %s", cudaGetErrorString(cudaError_t(rc))));
        }
        if (gframed) {
            // patch the request ids (known only after the fetch), expand this batch's stream descriptors, run K2
            for (size_t j = g0; j < g1; j++) sd[j].req_id = req_ids[j];
            cudaError_t ce = cudaMemcpyAsync(d_streams + g0, &sd[g0], sizeof(CvStreamDesc) * (g1 - g0), cudaMemcpyHostToDevice, G.vstream);
            const uint32_t fr0 = first_frame[g0], nfr = first_frame[g1] - fr0;
            int rc = ce != cudaSuccess ? int(ce) : 0;
            if (!rc) rc = cvk_expand_streams(d_streams + g0, static_cast<uint32_t>(g1 - g0), d_fdesc, first_frame[J], G.vstream);
            if (!rc && nfr)
                rc = cvk_unpack_frames(G.d_stage, d_fdesc + fr0, nfr, static_cast<uint32_t>(g1 - g0), d_dst, poly, gbytes,
                                       bc.verify ? d_crc + g0 : nullptr, d_ferr + fr0, G.vstream);
            if (rc) verr = Err::io(str_printf("cvk_unpack_frames: %s", cudaGetErrorString(cudaError_t(rc))));
            for (size_t g = v0; g < v1; g++)
                if (group_verbatim[g]) {
                    cudaEventRecord(G.free_ev[g % NS], G.vstream);
                    released[g % NS].store(static_cast<int64_t>(g), std::memory_order_release);
                }
        }
    }
    if (verr) st.fail(verr);
    for (auto& th : threads) th.join();
    if (st.err) {
        cudaStreamSynchronize(G.vstream);
        for (auto s : G.copy_streams) cudaStreamSynchronize(s);
        return st.err;
    }
    if (compare)
        CVK_TRY(cvk_verify_crcs_masked(d_crc + f0, reinterpret_cast<const uint32_t*>(T + o_exp) + f0, T + o_skip + f0, static_cast<uint32_t>(f1 - f0), d_crc + J, nullptr,
                                       G.vstream));
    if (n_segs)  // every copy group was waited for and CRC'd on vstream by now: scatter the landed bytes into the page buffers
        CVK_TRY(cvk_gather_pages(d_dst, reinterpret_cast<const CvSeg*>(T + o_segs), static_cast<uint32_t>(n_segs), static_cast<uint64_t>(pages->total), pages->d_page_base,
                                 G.vstream));
    CU_TRY(cudaMemcpyAsync(G.h_result, d_crc, 4 * res_words, cudaMemcpyDeviceToHost, G.vstream));
    CU_TRY(cudaEventRecord(G.done_ev, G.vstream));
    CU_TRY(cudaStreamWaitEvent(static_cast<cudaStream_t>(user_stream), G.done_ev, 0));
    pending_.active = true, pending_.jobs = J, pending_.frames = F;
    pending_.f0 = bc.verify ? f0 : 0, pending_.f1 = bc.verify ? f1 : 0, pending_.n_compared = compare ? n_compared : 0;
    G.pending_owner = this;
    for (size_t j = 0; j < J; j++) stats_.bytes += h_len[j];
    stats_.blocks += J;
    stats_.kernel_launches += cvk_launch_count() - launches0;
    for (int t = 0; t < T_threads; t++) stats_.fetch_sec += fetch_sec[static_cast<size_t>(t)], stats_.h2d_bytes += h2d[static_cast<size_t>(t)];
    stats_.wall_sec += now_sec() - t_start;
    stats_.reg_hits = G.reg.hits.load(), stats_.reg_misses = G.reg.misses.load();
    stats_.reg_rejected = G.reg.rejected.load(), stats_.reg_bytes = G.reg.bytes();
    stats_.ring_alloc_sec = G.ring_alloc_sec;
    stats_.gds_bytes += gds_bytes.load();
    return Err::ok();
}

Err GpuFsReader::read_many(FsContext* ctx, const std::vector<std::string>& paths, const int64_t* dst_offs, void* d_dst, int64_t cap, void* stream,
                            uint64_t* sum_crc, uint32_t* n_bad, uint64_t* n_verified, int64_t* total_bytes) {
    std::unique_ptr<GpuFsReader> r(new GpuFsReader());
    r->ctx_ = ctx;
    Err e;
    r->ing_ = gpu_ingest_get(ctx, &e);
    if (e) return e;
    std::vector<Job> jobs;
    int64_t total = 0;
    for (size_t i = 0; i < paths.size(); i++) {
        std::shared_ptr<const FileBlocks> fb;
        CV_RETURN_IF_ERR(ctx->ns.get_block_locations(paths[i], &fb));
        r->held_files_.push_back(fb);
        if (dst_offs[i] < 0 || dst_offs[i] + fb->status.len > cap) return Err::common("destination too small for " + paths[i]);
        for (size_t b = 0; b < fb->block_locs.size(); b++) {
            const int64_t blen = fb->block_locs[b].block.len;
            if (blen > 0) jobs.push_back(Job{&fb->block_locs[b], 0, blen, dst_offs[i] + fb->starts[b], true});
        }
        total += fb->status.len;
    }
    if (!r->held_files_.empty()) r->fbp_ = r->held_files_[0];
    CV_RETURN_IF_ERR(r->run_jobs(jobs, static_cast<uint8_t*>(d_dst), stream));
    if (total_bytes) *total_bytes = total;
    return r->verify(sum_crc, n_bad, n_verified);
}

}  // namespace cv
