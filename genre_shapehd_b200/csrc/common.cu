// common.cu — error plumbing of the C ABI.
#include "common.cuh"
#include <string.h>

namespace gb {
static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int fail_arg(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
int check_launch(const char *what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e == cudaSuccess) return 0;
  cudaGetLastError();  // clear the launch error so the next call starts clean
  set_error("%s: %s", what, cudaGetErrorString(e));
  return (int)e;
}
const char *last_error() { return g_err; }
}  // namespace gb

extern "C" const char *genre_b200_last_error(void) { return gb::last_error(); }
extern "C" int genre_b200_version(void) { return 2001; }
