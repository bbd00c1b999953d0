// api.cu -- error reporting and ABI self-description for libnmarl.
#include <stdarg.h>
#include <new>
#include "bwd_common.cuh"

static thread_local char g_err[512] = "";

void nmarl_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* nmarl_last_error(void) { return g_err; }
extern "C" int nmarl_version(void) { return 101; }
extern "C" int nmarl_sizeof_model(void) { return (int)sizeof(nmarl_model); }
extern "C" int nmarl_sizeof_agent(void) { return (int)sizeof(nmarl_agent); }
extern "C" int nmarl_sizeof_cacc_cfg(void) { return (int)sizeof(nmarl_cacc_cfg); }
extern "C" int nmarl_sizeof_fwd_args(void) { return (int)sizeof(nmarl_fwd_args); }
extern "C" int nmarl_sizeof_bwd_args(void) { return (int)sizeof(nmarl_bwd_args); }

extern "C" int nmarl_create(nmarl_ctx** out) {
  NMARL_CHECK(out != nullptr, "nmarl_create: out is NULL");
  nmarl_ctx* c = new (std::nothrow) nmarl_ctx();
  NMARL_CHECK(c != nullptr, "nmarl_create: out of host memory");
  c->side = nullptr; c->fork = nullptr; c->join = nullptr; c->heads = nullptr;
  cudaError_t e = cudaGetDevice(&c->device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->heads, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    nmarl_set_error("nmarl_create: %s", cudaGetErrorString(e));
    nmarl_destroy(c);
    return 2;
  }
  *out = c;
  return 0;
}

extern "C" int nmarl_destroy(nmarl_ctx* c) {
  if (c == nullptr) return 0;
  if (c->fork) cudaEventDestroy(c->fork);
  if (c->join) cudaEventDestroy(c->join);
  if (c->heads) cudaEventDestroy(c->heads);
  if (c->side) cudaStreamDestroy(c->side);
  delete c;
  return 0;
}

// debug hook (not part of the public ABI): device buffer of >= 128 int64 receiving clock64() stamps from
// CTA (0,0) of the tensor-core forward kernel
long long* g_nmarl_prof = nullptr;
extern "C" __attribute__((visibility("default"))) void nmarl_debug_set_prof(long long* p) { g_nmarl_prof = p; }
