// errors.cu -- status / error-string plumbing of the C ABI (include/spacap3d_ops.h).
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace spc {
static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what) {
  set_error("CUDA error %d (%s) at: %s", (int)e, cudaGetErrorString(e), what);
  return SPC_ERR_CUDA;
}
}  // namespace spc

extern "C" int spc_abi_version(void) { return 20; }
extern "C" const char *spc_last_error(void) { return spc::g_err; }
