// Library-level plumbing of libhicgat_sm100.so: version, thread-local error text, launch counter.
#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "common.cuh"

namespace hicgat {
namespace {
thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
}  // namespace

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }
}  // namespace hicgat

extern "C" int hicgat_version(void) { return 202; }
extern "C" const char* hicgat_last_error(void) { return hicgat::g_err; }
extern "C" uint64_t hicgat_launch_count(void) { return hicgat::g_launches.load(std::memory_order_relaxed); }

// Strided host -> device copy on the caller's stream (cudaMemcpy2DAsync): the host-buffer loss path of a SYMMETRIC target
// uploads only the columns at or right of a row block's diagonal, i.e. a sub-rectangle of the pinned host matrix.
extern "C" int hicgat_memcpy2d_h2d_async(void* dst_device, size_t dst_pitch_bytes, const void* src_host, size_t src_pitch_bytes,
                                         size_t width_bytes, size_t height, hicgat_stream_t stream) {
    using namespace hicgat;
    HICGAT_REQUIRE(dst_device && src_host && width_bytes <= dst_pitch_bytes && width_bytes <= src_pitch_bytes, "hicgat_memcpy2d_h2d_async: bad arguments");
    if (width_bytes == 0 || height == 0) return HICGAT_OK;
    HICGAT_CUDA(cudaMemcpy2DAsync(dst_device, dst_pitch_bytes, src_host, src_pitch_bytes, width_bytes, height, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
    return HICGAT_OK;
}
