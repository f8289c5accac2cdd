// api.cu -- library-level entry points of libtmf_sm100a (error string, device gate, launch counter).
#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "common.cuh"

namespace tmf {

static thread_local char g_err[1024] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

}  // namespace tmf

extern "C" {

const char* tmf_last_error(void) { return tmf::g_err; }

int tmf_version(void) { return 200; }

int tmf_stat_rows(void) { return TMF_STAT_ROWS; }

int64_t tmf_launch_count(void) { return tmf::g_launches.load(std::memory_order_relaxed); }

int tmf_check_device(void) {
  int dev = 0;
  TMF_CUDA(cudaGetDevice(&dev));
  int major = 0, minor = 0;
  TMF_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  TMF_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  TMF_REQUIRE(major == 10, "libtmf_sm100a is built for sm_100a only; device %d is cc %d.%d (no fallback path)", dev,
              major, minor);
  return 0;
}

}  // extern "C"
