// Library-level entry points: error reporting, version, device queries.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include <atomic>
#include "common.cuh"
#include "serl_b200.h"

namespace serl {

static thread_local char g_err[512] = "";

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<unsigned long long> g_launches{0};

// Every launcher calls this exactly once after its <<<...>>> (the only other call sites are cudaFuncSetAttribute failure
// paths), so the number of successful checks is the number of kernels this library has enqueued.
int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_last_error("%s: %s", what, cudaGetErrorString(e));
    return SERL_ERR_CUDA;
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return SERL_OK;
}
unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

static int g_pdl = -1;
bool pdl_enabled() {
  if (g_pdl < 0) { const char* e = getenv("SERL_PDL"); g_pdl = (e && atoi(e) != 0) ? 1 : 0; }
  return g_pdl != 0;
}

}  // namespace serl

extern "C" const char* serl_last_error(void) { return serl::g_err; }
namespace serl {
int balanced_grid(int items, int sms) {
  static int full = -1;
  if (full < 0) { const char* e = getenv("SERL_FULL_GRID"); full = (e && atoi(e) != 0) ? 1 : 0; }
  static int limit = -1;                                          // SERL_TRUNK_SM_LIMIT=n: at most n CTAs (experiments: SM share of the trunk)
  if (limit < 0) { const char* e = getenv("SERL_TRUNK_SM_LIMIT"); limit = e ? atoi(e) : 0; }
  if (limit > 0 && limit < sms) sms = limit;
  if (items <= sms || full) return items < sms ? items : sms;
  const int waves = (items + sms - 1) / sms;
  return (items + waves - 1) / waves;
}
}  // namespace serl

extern "C" int serl_balanced_grid(int items, int sms) { return serl::balanced_grid(items, sms); }
extern "C" int serl_version(void) { return 4; }
extern "C" unsigned long long serl_launch_count(void) { return serl::launch_count(); }
extern "C" int serl_set_pdl(int enabled) { serl::g_pdl = enabled ? 1 : 0; return SERL_OK; }
extern "C" int serl_device_sm_count(int device) {
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) {
    serl::set_last_error("serl_device_sm_count: no CUDA device %d", device);
    return SERL_ERR_CUDA;
  }
  return n;
}
