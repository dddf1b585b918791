// GPUDirect Storage for the SSD/HDD tiers (SURVEY.md 8f-2): cuFileRead straight into the destination in HBM, no pinned host
// ring in between.  libcufile is dlopen'ed at first use (the product library carries no link-time dependency on it); when it is
// missing, when the driver cannot be opened, or when a file cannot be registered, the caller falls back to the pinned ring and
// says so in the read stats.  Only real GPUDirect Storage is used: without the nvidia-fs kernel module cuFile could only run in its
// compatibility mode (POSIX reads into its own pinned bounce buffers + copies), which the pinned ring outruns, so libcufile is then
// not loaded at all.
#pragma once
#include "common.h"

namespace cv {

struct GdsInfo {
    bool available = false;  // libcufile loaded and cuFileDriverOpen succeeded
    bool compat = false;     // no nvidia-fs kernel module: cuFile would only have its compatibility mode, and is not opened
    std::string detail;
};

// Probes once per process.  Without the nvidia-fs module cuFile is not opened at all: available = false, compat = true.
const GdsInfo& gds_info();
// n bytes of `path` starting at file_off -> d_dst (device memory of the current device).  kUnsupported when GDS cannot serve it.
Err gds_read(const std::string& path, void* d_dst, int64_t n, int64_t file_off);
std::string gds_last_refusal();  // why the first file that was turned away was turned away ("" if none was)
void gds_forget(const std::string& path);  // drop the cached handle (file replaced / context teardown: "" = all)

}  // namespace cv
