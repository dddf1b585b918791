#include "gds.h"

#include <dlfcn.h>
#include <errno.h>
#include <fcntl.h>
#include <stdlib.h>
#include <sys/stat.h>
#include <unistd.h>

#include <mutex>
#include <unordered_map>

// The handful of cuFile declarations used here (cufile.h, CUDA 12.x ABI), restated so that this file needs neither the header
// nor the library at build time.
extern "C" {
typedef struct {
    int err;     // CUfileOpError; 0 == CU_FILE_SUCCESS
    int cu_err;  // CUresult
} CvCuFileError;
typedef void* CvCuFileHandle;
typedef struct {
    int type;  // 1 == CU_FILE_HANDLE_TYPE_OPAQUE_FD
    union {
        int fd;
        void* handle;
    } handle;
    const void* fs_ops;
} CvCuFileDescr;
}

namespace cv {
namespace {

struct Api {
    void* lib = nullptr;
    CvCuFileError (*DriverOpen)() = nullptr;
    CvCuFileError (*HandleRegister)(CvCuFileHandle*, CvCuFileDescr*) = nullptr;
    void (*HandleDeregister)(CvCuFileHandle) = nullptr;
    ssize_t (*Read)(CvCuFileHandle, void*, size_t, off_t, off_t) = nullptr;
};

struct Entry {
    int fd = -1;
    CvCuFileHandle h = nullptr;
    uint64_t ino = 0;
};

std::once_flag g_once;
Api g_api;
GdsInfo g_info;
std::mutex g_mu;
std::unordered_map<std::string, Entry> g_files;

std::string g_refusal;  // first reason a file was turned away (under g_mu)

bool nvidia_fs_loaded() {
    return access("/proc/driver/nvidia-fs/stats", R_OK) == 0;  // the nvidia-fs module publishes this file
}

void probe() {
    const char* names[] = {"libcufile.so.0", "libcufile.so", "/usr/local/cuda/lib64/libcufile.so.0", "/usr/local/cuda/lib64/libcufile.so"};
    for (const char* n : names)
        if ((g_api.lib = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
    if (!g_api.lib) {
        g_info.detail = "libcufile not found";
        return;
    }
    g_api.DriverOpen = reinterpret_cast<decltype(g_api.DriverOpen)>(dlsym(g_api.lib, "cuFileDriverOpen"));
    g_api.HandleRegister = reinterpret_cast<decltype(g_api.HandleRegister)>(dlsym(g_api.lib, "cuFileHandleRegister"));
    g_api.HandleDeregister = reinterpret_cast<decltype(g_api.HandleDeregister)>(dlsym(g_api.lib, "cuFileHandleDeregister"));
    g_api.Read = reinterpret_cast<decltype(g_api.Read)>(dlsym(g_api.lib, "cuFileRead"));
    if (!g_api.DriverOpen || !g_api.HandleRegister || !g_api.HandleDeregister || !g_api.Read) {
        g_info.detail = "libcufile lacks an expected symbol";
        return;
    }
    const CvCuFileError e = g_api.DriverOpen();
    if (e.err != 0) {
        g_info.detail = str_printf("cuFileDriverOpen failed: cufile error %d, cuda error %d", e.err, e.cu_err);
        return;
    }
    g_info.available = true;
    g_info.detail = "GPUDirect Storage (nvidia-fs)";
}

}  // namespace

const GdsInfo& gds_info() {
    // Without nvidia-fs cuFile could only run in its compatibility mode, which is slower than the pinned ring; and opening cuFile's
    // driver on a B200 without nvidia-fs stalled the first short-circuit read of a process for more than three minutes (observed in
    // one test run).  The library is then not loaded at all.
    static const bool native = nvidia_fs_loaded();
    if (!native) {
        static const GdsInfo closed{false, true, "nvidia-fs kernel module not loaded: cuFile is not opened, disk-tier blocks take the pinned ring"};
        return closed;
    }
    std::call_once(g_once, probe);
    return g_info;
}

std::string gds_last_refusal() {
    std::lock_guard<std::mutex> lk(g_mu);
    return g_refusal;
}

void gds_forget(const std::string& path) {
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto it = g_files.begin(); it != g_files.end();) {
        if (path.empty() || it->first == path) {
            if (it->second.h) g_api.HandleDeregister(it->second.h);
            if (it->second.fd >= 0) ::close(it->second.fd);
            it = g_files.erase(it);
        } else {
            ++it;
        }
    }
}

Err gds_read(const std::string& path, void* d_dst, int64_t n, int64_t file_off) {
    const GdsInfo& gi = gds_info();
    if (!gi.available) return Err(kUnsupported, "GDS unavailable: " + gi.detail);
    Entry e;
    {
        struct stat st;
        if (stat(path.c_str(), &st) != 0) return Err::io(str_printf("stat %s: %s", path.c_str(), strerror(errno)));
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_files.find(path);
        if (it != g_files.end() && it->second.ino != static_cast<uint64_t>(st.st_ino)) {  // the block file was replaced
            g_api.HandleDeregister(it->second.h);
            ::close(it->second.fd);
            g_files.erase(it);
            it = g_files.end();
        }
        if (it == g_files.end()) {
            Entry ne;
            // GDS wants O_DIRECT; a file system that refuses it gets a plain descriptor, and cuFileHandleRegister decides
            ne.fd = ::open(path.c_str(), O_RDONLY | O_DIRECT | O_CLOEXEC);
            if (ne.fd < 0) ne.fd = ::open(path.c_str(), O_RDONLY | O_CLOEXEC);
            if (ne.fd < 0) return Err::io(str_printf("open %s: %s", path.c_str(), strerror(errno)));
            CvCuFileDescr d;
            memset(&d, 0, sizeof(d));
            d.type = 1, d.handle.fd = ne.fd;
            const CvCuFileError ce = g_api.HandleRegister(&ne.h, &d);
            if (ce.err != 0) {
                ::close(ne.fd);
                Err e(kUnsupported, str_printf("cuFileHandleRegister(%s): cufile error %d, cuda error %d", path.c_str(), ce.err, ce.cu_err));
                if (g_refusal.empty()) g_refusal = e.msg;
                return e;
            }
            ne.ino = static_cast<uint64_t>(st.st_ino);
            it = g_files.emplace(path, ne).first;
        }
        e = it->second;
    }
    int64_t got = 0;
    while (got < n) {
        const ssize_t r = g_api.Read(e.h, d_dst, static_cast<size_t>(n - got), static_cast<off_t>(file_off + got), static_cast<off_t>(got));
        if (r < 0) return Err::io(str_printf("cuFileRead(%s): %zd (errno %d)", path.c_str(), r, errno));
        if (r == 0) return Err::io("cuFileRead: unexpected end of file");
        got += r;
    }
    return Err::ok();
}

}  // namespace cv
