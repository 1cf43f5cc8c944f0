// md2_capi.cu - extern "C" boundary of libmd2loss.so (declared in include/md2_loss.h).
#include <cuda_runtime.h>

#include "../../include/md2_loss.h"
#include "md2_core.cuh"
#include "md2_plan.h"

namespace md2 {
#if defined(MD2_DBG_DEVICE) || defined(MD2_BOUNDS_CHECK)
cudaError_t debug_set_sink(const DebugSink* host_copy);
cudaError_t debug_oob_count(unsigned long long* count, int reset);
#endif
cudaError_t launch_view_synthesis_loss(const Params& P, const Widen& Wd, cudaStream_t stream);
cudaError_t profile_enable(bool on);
cudaError_t profile_march_ms(float* ms);
}

extern "C" {

int md2_version(void) { return 101; }

const char* md2_status_string(int status) {
  switch (status) {
    case MD2_OK: return "ok";
    case MD2_ERR_INVALID_ARGUMENT: return "invalid argument";
    case MD2_ERR_UNSUPPORTED: return "unsupported configuration";
    case MD2_ERR_WORKSPACE_TOO_SMALL: return "workspace too small";
    case MD2_ERR_CUDA: return "CUDA error";
    default: return "unknown status";
  }
}

int md2_loss_workspace_bytes(const md2_problem* p, size_t* bytes) {
  if (!bytes) return MD2_ERR_INVALID_ARGUMENT;
  const int st = md2::validate(p);
  if (st != MD2_OK) return st;
  *bytes = md2::make_layout(p).total;
  return MD2_OK;
}

int md2_view_synthesis_loss(const md2_problem* p, const md2_tensors* t, void* workspace,
                            size_t workspace_bytes, void* stream) {
  int st = md2::validate(p);
  if (st != MD2_OK) return st;
  if (workspace_bytes < md2::make_layout(p).total) return MD2_ERR_WORKSPACE_TOO_SMALL;
  md2::Params P;
  st = md2::fill_params(p, t, workspace, &P);
  if (st != MD2_OK) return st;
  md2::Widen Wd;
  md2::fill_widen(p, workspace, &P, &Wd);
  const cudaError_t e = md2::launch_view_synthesis_loss(P, Wd, (cudaStream_t)stream);
  return e == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

int md2_profile_enable(int on) {
  return md2::profile_enable(on != 0) == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

int md2_profile_march_ms(float* ms) {
  if (!ms) return MD2_ERR_INVALID_ARGUMENT;
  return md2::profile_march_ms(ms) == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}

#if defined(MD2_DBG_DEVICE) || defined(MD2_BOUNDS_CHECK)
/* debug build only (libmd2loss_dbg.so, include/md2_debug.h): decision export + bounds-check counter */
int md2_debug_set_sink(const void* sink) {
  return md2::debug_set_sink((const md2::DebugSink*)sink) == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}
int md2_debug_oob_count(unsigned long long* count, int reset) {
  if (!count) return MD2_ERR_INVALID_ARGUMENT;
  return md2::debug_oob_count(count, reset) == cudaSuccess ? MD2_OK : MD2_ERR_CUDA;
}
#endif

}  // extern "C"
