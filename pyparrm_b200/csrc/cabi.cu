// Library-level entry points of libparrm_b200: version, error string, device probe,
// and the FP64 FMA burn used by bench.py to measure the evaluator's roofline peak.
#include <stdarg.h>

#include "common.cuh"

namespace parrm {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

// Each thread runs 8 independent DFMA chains of `iters` steps (2 flops each).
__global__ void __launch_bounds__(256) fp64_burn_kernel(int64_t iters, double* sink) {
  double a0 = 1.0 + threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
  double a4 = a0 + 4e-3, a5 = a0 + 5e-3, a6 = a0 + 6e-3, a7 = a0 + 7e-3;
  const double m = 0.999999999, c = 1e-9;
  for (int64_t i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (s == 123.456) sink[0] = s;  // never true; keeps the chains alive
}

template <typename S, typename D>
__global__ void __launch_bounds__(256) convert_kernel(const S* __restrict__ src,
                                                      D* __restrict__ dst, int64_t n) {
  for (int64_t i = int64_t(blockIdx.x) * 256 + threadIdx.x; i < n; i += int64_t(gridDim.x) * 256)
    dst[i] = static_cast<D>(src[i]);
}

template <typename S, typename D>
int convert(const S* src, D* dst, int64_t n, void* stream, const char* name) {
  if (n <= 0) return PARRM_OK;
  if (src == nullptr || dst == nullptr) {
    set_error("%s: null pointer", name);
    return PARRM_ERR_INVALID_ARGUMENT;
  }
  const int64_t blocks = min64(ceil_div(n, 256), int64_t(kNumSMs) * 16);
  convert_kernel<S, D><<<unsigned(blocks), 256, 0, as_stream(stream)>>>(src, dst, n);
  PARRM_LAUNCH_OK(name);
  return PARRM_OK;
}

// Storage types a recording may arrive in (parrm_storage_t): the reference accepts any 2-D
// ndarray (parrm.py:877-886) and widens it on the host; here the caller's bytes cross PCIe as
// they are and are widened on the device.
template <typename S>
int convert_from(const S* src, void* d_dst, int dst_type, int64_t n, void* stream) {
  if (dst_type == PARRM_F64)
    return convert<S, double>(src, static_cast<double*>(d_dst), n, stream, "parrm_convert");
  if (dst_type == PARRM_F32)
    return convert<S, float>(src, static_cast<float*>(d_dst), n, stream, "parrm_convert");
  set_error("parrm_convert: destination must be float64 or float32");
  return PARRM_ERR_INVALID_ARGUMENT;
}

}  // namespace parrm

extern "C" {

int parrm_convert_f64_to_f32(const double* d_src, float* d_dst, int64_t n, void* stream) {
  return parrm::convert<double, float>(d_src, d_dst, n, stream, "parrm_convert_f64_to_f32");
}

int parrm_convert_f32_to_f64(const float* d_src, double* d_dst, int64_t n, void* stream) {
  return parrm::convert<float, double>(d_src, d_dst, n, stream, "parrm_convert_f32_to_f64");
}

int parrm_convert(const void* d_src, int src_type, void* d_dst, int dst_type, int64_t n,
                  void* stream) {
  switch (src_type) {
    case PARRM_F64: return parrm::convert_from(static_cast<const double*>(d_src), d_dst, dst_type, n, stream);
    case PARRM_F32: return parrm::convert_from(static_cast<const float*>(d_src), d_dst, dst_type, n, stream);
    case PARRM_I16: return parrm::convert_from(static_cast<const int16_t*>(d_src), d_dst, dst_type, n, stream);
    case PARRM_I32: return parrm::convert_from(static_cast<const int32_t*>(d_src), d_dst, dst_type, n, stream);
    default:
      parrm::set_error("parrm_convert: unknown source type %d", src_type);
      return PARRM_ERR_INVALID_ARGUMENT;
  }
}

int parrm_host_register(void* h_ptr, size_t bytes) {
  PARRM_REQUIRE(h_ptr != nullptr && bytes > 0, "parrm_host_register: empty range");
  PARRM_CUDA_OK(cudaHostRegister(h_ptr, bytes, cudaHostRegisterPortable));
  return PARRM_OK;
}

int parrm_host_unregister(void* h_ptr) {
  PARRM_REQUIRE(h_ptr != nullptr, "parrm_host_unregister: null pointer");
  PARRM_CUDA_OK(cudaHostUnregister(h_ptr));
  return PARRM_OK;
}

int parrm_abi_version(void) { return PARRM_B200_ABI_VERSION; }

const char* parrm_last_error(void) { return parrm::g_error; }

int parrm_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int parrm_host_is_pinned(const void* h_ptr) {
  if (h_ptr == nullptr) return 0;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, h_ptr) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return attr.type == cudaMemoryTypeHost ? 1 : 0;
}

int parrm_copy_h2d_async(void* d_dst, const void* h_src, size_t bytes, void* stream) {
  if (bytes == 0) return PARRM_OK;
  PARRM_REQUIRE(d_dst && h_src, "parrm_copy_h2d_async: null pointer");
  PARRM_CUDA_OK(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice,
                                parrm::as_stream(stream)));
  return PARRM_OK;
}

int parrm_copy_d2h_async(void* h_dst, const void* d_src, size_t bytes, void* stream) {
  if (bytes == 0) return PARRM_OK;
  PARRM_REQUIRE(h_dst && d_src, "parrm_copy_d2h_async: null pointer");
  PARRM_CUDA_OK(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost,
                                parrm::as_stream(stream)));
  return PARRM_OK;
}

int parrm_copy_h2d_2d_async(void* d_dst, size_t dst_pitch, const void* h_src, size_t src_pitch,
                            size_t width, size_t height, void* stream) {
  if (width == 0 || height == 0) return PARRM_OK;
  PARRM_REQUIRE(d_dst && h_src, "parrm_copy_h2d_2d_async: null pointer");
  PARRM_REQUIRE(dst_pitch >= width && src_pitch >= width,
                "parrm_copy_h2d_2d_async: pitch below the row width");
  PARRM_CUDA_OK(cudaMemcpy2DAsync(d_dst, dst_pitch, h_src, src_pitch, width, height,
                                  cudaMemcpyHostToDevice, parrm::as_stream(stream)));
  return PARRM_OK;
}

int parrm_copy_d2h_2d_async(void* h_dst, size_t dst_pitch, const void* d_src, size_t src_pitch,
                            size_t width, size_t height, void* stream) {
  if (width == 0 || height == 0) return PARRM_OK;
  PARRM_REQUIRE(h_dst && d_src, "parrm_copy_d2h_2d_async: null pointer");
  PARRM_REQUIRE(dst_pitch >= width && src_pitch >= width,
                "parrm_copy_d2h_2d_async: pitch below the row width");
  PARRM_CUDA_OK(cudaMemcpy2DAsync(h_dst, dst_pitch, d_src, src_pitch, width, height,
                                  cudaMemcpyDeviceToHost, parrm::as_stream(stream)));
  return PARRM_OK;
}

int parrm_fp64_fma_burn(int64_t iters, double* d_sink, double* h_flops, void* stream) {
  PARRM_REQUIRE(iters > 0 && d_sink != nullptr, "parrm_fp64_fma_burn: bad arguments");
  const int blocks = parrm::kNumSMs * 8, threads = 256;
  parrm::fp64_burn_kernel<<<blocks, threads, 0, parrm::as_stream(stream)>>>(iters, d_sink);
  PARRM_LAUNCH_OK("fp64_burn_kernel");
  if (h_flops) *h_flops = 2.0 * 8.0 * double(iters) * double(blocks) * double(threads);
  return PARRM_OK;
}

}  // extern "C"
