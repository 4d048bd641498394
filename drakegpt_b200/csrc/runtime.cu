// Error plumbing, device gate and small host-side utilities of the C-ABI.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace dgpt {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return DGPT_E_LAUNCH;
  }
  return DGPT_OK;
}

unsigned long long* clock_probe_buffer() {
  static int on = -1;
  static unsigned long long* buf = nullptr;
  if (on < 0) {
    const char* e = getenv("DGPT_CLOCK_PROBE");
    on = e ? (atoi(e) != 0) : 0;
    if (on && cudaMalloc(&buf, 64 * sizeof(unsigned long long)) != cudaSuccess) { cudaGetLastError(); buf = nullptr; }
  }
  return buf;
}

bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DGPT_PDL");
    v = e ? (atoi(e) != 0) : 1;
  }
  return v != 0;
}

// One probe per device per process; there is no CPU fallback behind this gate.
int require_device() {
  static thread_local int cached_dev = -1;
  static thread_local int cached_rc = 0;
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("no CUDA device: %s (drakegpt_b200 has no CPU fallback)", cudaGetErrorString(e));
    return DGPT_E_DEVICE;
  }
  if (dev == cached_dev) return cached_rc;
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess || major != 10) {
    cudaGetLastError();
    set_error("device %d has compute capability major %d; kernels are built for sm_100a only", dev,
              major);
    cached_dev = dev;
    cached_rc = DGPT_E_DEVICE;
    return cached_rc;
  }
  cached_dev = dev;
  cached_rc = DGPT_OK;
  return DGPT_OK;
}

}  // namespace dgpt

extern "C" {

const char* dgpt_last_error(void) { return dgpt::g_err; }
int dgpt_abi_version(void) { return 2; }

int dgpt_device_check(void) { return dgpt::require_device(); }

int dgpt_sm_count(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return DGPT_E_DEVICE;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return DGPT_E_DEVICE;
  return n;
}

/* (cycles, nanoseconds) between entry and exit of CTA 0 of the last kernel launched with DGPT_CLOCK_PROBE=1 */
int dgpt_debug_clock_probe(uint64_t* cycles, uint64_t* ns) {
  unsigned long long h[4] = {0, 0, 0, 0};
  unsigned long long* buf = dgpt::clock_probe_buffer();
  if (!buf) { dgpt::set_error("clock probe is off (DGPT_CLOCK_PROBE=1 enables it)"); return DGPT_E_ARG; }
  if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpy(h, buf, sizeof(h), cudaMemcpyDeviceToHost) != cudaSuccess) {
    cudaGetLastError();
    return DGPT_E_DEVICE;
  }
  *cycles = h[2] - h[0];
  *ns = h[3] - h[1];
  return DGPT_OK;
}

/* the raw 64-word stamp buffer (words 0-3 as above, 4.. = kernel-specific phase stamps in cycles) */
int dgpt_debug_clock_stamps(uint64_t* out64) {
  unsigned long long* buf = dgpt::clock_probe_buffer();
  if (!buf) { dgpt::set_error("clock probe is off (DGPT_CLOCK_PROBE=1 enables it)"); return DGPT_E_ARG; }
  if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpy(out64, buf, 64 * sizeof(uint64_t), cudaMemcpyDeviceToHost) != cudaSuccess) {
    cudaGetLastError();
    return DGPT_E_DEVICE;
  }
  return DGPT_OK;
}

int dgpt_dropout_keep_host(uint64_t seed, uint32_t site, uint64_t index, float p) {
  return dgpt::dropout_keep(seed, site, index, dgpt::dropout_threshold(p)) ? 1 : 0;
}

}  // extern "C"
