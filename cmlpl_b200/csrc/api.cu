// Error plumbing, device queries and the per-device side stream for the C ABI (include/cmlpl.h).
#include <stdarg.h>
#include <string.h>

#include <cudaTypedefs.h>

#include "common.cuh"
#include "tma.cuh"

namespace cmlpl {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
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

SideStream* side_stream() {
  static SideStream per_dev[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  SideStream& x = per_dev[dev];
  std::lock_guard<std::mutex> lock(x.mu);
  if (x.s) return &x;
  // complete or nothing: a failed creation releases what it made and leaves the slot empty for the next call
  cudaStream_t s = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  bool ok = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess;
  for (cudaEvent_t& e : ev) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    for (cudaEvent_t e : ev)
      if (e) cudaEventDestroy(e);
    if (s) cudaStreamDestroy(s);
    return nullptr;
  }
  x.fork[0] = ev[0]; x.join[0] = ev[1]; x.fork[1] = ev[2]; x.join[1] = ev[3];
  x.s = s;
  return &x;
}

int make_scene_tmap(CUtensorMap* out, const void* base, int outer, int rows, int cols, int box_rows, int box_cols) {
  static PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
        qres != cudaDriverEntryPointSuccess) {
      set_error("cuTensorMapEncodeTiled entry point not available");
      return CMLPL_ERR_CUDA;
    }
    encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  }
  const cuuint64_t psz = cuuint64_t(rows) * cols;
  // a row of the plane is contiguous (cols x 16 B), so (8 halves, cols) is ONE dimension of cols*8 halves: the box's
  // innermost extent is box_cols*16 bytes (512 B for 32 columns) instead of 16 B, which is what the TMA unit likes
  const cuuint64_t dims[4] = {cuuint64_t(cols) * 8, cuuint64_t(rows), 8, cuuint64_t(outer)};
  const cuuint64_t strides[3] = {cuuint64_t(cols) * 16, psz * 16, psz * 128};       // bytes, dims 1..3
  const cuuint32_t box[4] = {cuuint32_t(box_cols) * 8, cuuint32_t(box_rows), 8, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for [%d][8][%d][%d][8] box %dx%d", int(r), outer, rows, cols, box_rows, box_cols);
    return CMLPL_ERR_CUDA;
  }
  return CMLPL_OK;
}

}  // namespace cmlpl

extern "C" {

int cmlpl_version(void) { return 101; }

const char* cmlpl_last_error(void) { return cmlpl::g_err; }

int cmlpl_device_ok(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cmlpl::set_error("cmlpl_device_ok: no CUDA device");
    return CMLPL_ERR_CUDA;
  }
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  return (major == 10 && minor == 0) ? 1 : 0;
}

int cmlpl_memcpy2d_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes, size_t height,
                         cmlpl_stream_t stream) {
  CMLPL_CHECK_ARG(dst && src, "memcpy2d_async: null pointer");
  CMLPL_CHECK_ARG(width_bytes <= dpitch && width_bytes <= spitch, "memcpy2d_async: width %zu exceeds a pitch (%zu, %zu)",
                  width_bytes, dpitch, spitch);
  if (width_bytes == 0 || height == 0) return CMLPL_OK;
  CMLPL_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width_bytes, height, cudaMemcpyDefault,
                               static_cast<cudaStream_t>(stream)));
  return CMLPL_OK;
}

}  // extern "C"
