// api_common.cu -- error reporting and device queries shared by every C-ABI entry point.
#include "common.cuh"

namespace g4r {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? G4R_ENODEVICE : G4R_ECUDA;
}

int num_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// SMs the persistent (one CTA per SM) GEMM kernels may occupy: all of them minus the reserve set through
// g4r_set_sm_reserve().  A collective running beside the backward (NCCL's CTAs are long-lived too) needs SMs of its
// own: if the GEMM grid covers every SM, its statically scheduled CTAs queue behind the collective's CTAs and the two
// serialise instead of overlapping.
static int g_sm_reserve = 0;
int sm_budget() {
  int n = num_sms() - g_sm_reserve;
  return n < 2 ? 2 : n;
}
void set_sm_reserve_impl(int n) { g_sm_reserve = n < 0 ? 0 : n; }

// Programmatic dependent launch is opt-in per call sequence (g4r_set_pdl): a kernel launched this way reads its
// weights BEFORE the predecessor kernel's writes are guaranteed visible, which is only sound when no kernel of the
// sequence writes them -- true for the decode step, not for arbitrary callers (a cast or an optimizer kernel may
// directly precede a small GEMM).
static int g_pdl_on = 0;
bool pdl_on() { return g_pdl_on != 0; }

}  // namespace g4r

extern "C" int g4r_set_pdl(int on) {
  const int prev = g4r::g_pdl_on;
  g4r::g_pdl_on = on ? 1 : 0;
  return prev;
}

extern "C" int g4r_set_sm_reserve(int n_sms) {
  const int prev = g4r::g_sm_reserve;
  g4r::set_sm_reserve_impl(n_sms);
  return prev;
}

extern "C" const char* g4r_last_error(void) { return g4r::g_err; }
extern "C" int g4r_version(void) { return 1001; }
extern "C" int g4r_built_arch(void) { return 100; }
