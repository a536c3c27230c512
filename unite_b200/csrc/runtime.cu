// Error plumbing and device queries shared by every C-ABI entry point.
#include "common.cuh"
#include "../../include/unite_b200.h"
#include <cstdarg>
#include <cstdio>

namespace ub {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
    return 1;
  }
  return 0;
}

static int g_sm_limit = 0;   // 0 = all SMs; otherwise the persistent grids leave the rest to a concurrent collective

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return (g_sm_limit > 0 && g_sm_limit < n) ? g_sm_limit : n;
}

}  // namespace ub

extern "C" int ub_version(void) { return 100; }
extern "C" const char* ub_last_error(void) { return ub::g_err; }
extern "C" int ub_sm_count(void) { return ub::sm_count(); }
extern "C" int ub_set_sm_limit(int n) {
  ub::g_sm_limit = n > 0 ? (n & ~1) : 0;     // even, so CTA pairs still tile it
  return ub::sm_count();
}
