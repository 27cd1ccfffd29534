// Transposing convert for time-major ("interleaved") recordings: raw electrophysiology is stored
// [times, channels] (SpikeGLX, Open Ephys, Intan, Blackrock), the filter and the search read
// [channels, times].  One pass turns a [rows, cols] source with row pitch src_ld into a
// [cols, rows] destination with row pitch dst_ld, converting each element with static_cast as
// convert_kernel (cabi.cu) does, so a transposed chunk holds the same bytes as a converted one.
//
// A CTA moves one 64 x 64 tile through shared memory: 256 threads read it row by row (64
// source columns = one full 128-byte line of int16, two of float32 / int32, four of float64)
// and write it column by column (64 destination elements per row).  The shared row pitch is
// padded so that a warp reading one tile column hits 32 different banks: 65 elements for 4- and
// 8-byte types, 66 for 2-byte ones (33 words).  Loads are scalar, so any source base works (a
// channel-subset view starts mid-line); edge tiles are masked.
#include "common.cuh"

namespace parrm {
namespace {

constexpr int kTile = 64;
constexpr int kThreads = 256;
constexpr int kRowsPerPass = kThreads / kTile;  // 4

template <typename S>
__host__ __device__ constexpr int tile_pitch() { return sizeof(S) == 2 ? kTile + 2 : kTile + 1; }

template <typename S, typename D>
__global__ void __launch_bounds__(kThreads)
transpose_kernel(const S* __restrict__ src, int64_t rows, int64_t cols, int64_t src_ld,
                 D* __restrict__ dst, int64_t dst_ld, int64_t col_tiles) {
  __shared__ S tile[kTile * tile_pitch<S>()];
  constexpr int P = tile_pitch<S>();
  const int lane = threadIdx.x % kTile, sub = threadIdx.x / kTile;
  const int64_t r0 = int64_t(blockIdx.x) * kTile;
  for (int64_t ct = blockIdx.y; ct < col_tiles; ct += gridDim.y) {
    const int64_t c0 = ct * kTile;
    // read: tile row i = source row r0 + i, lane = source column c0 + lane
    const int64_t c = c0 + lane;
#pragma unroll 4
    for (int i = sub; i < kTile; i += kRowsPerPass) {
      const int64_t r = r0 + i;
      if (r < rows && c < cols) tile[i * P + lane] = src[r * src_ld + c];
    }
    __syncthreads();
    // write: destination row c0 + j (a source column), lane = destination column r0 + lane
    const int64_t r = r0 + lane;
#pragma unroll 4
    for (int j = sub; j < kTile; j += kRowsPerPass) {
      const int64_t cj = c0 + j;
      if (r < rows && cj < cols) dst[cj * dst_ld + r] = static_cast<D>(tile[lane * P + j]);
    }
    __syncthreads();
  }
}

template <typename S, typename D>
int launch(const void* src, int64_t rows, int64_t cols, int64_t src_ld, void* dst,
           int64_t dst_ld, void* stream) {
  const int64_t row_tiles = ceil_div(rows, kTile), col_tiles = ceil_div(cols, kTile);
  PARRM_REQUIRE(row_tiles <= 0x7fffffff, "parrm_transpose: %lld rows is too many",
                (long long)rows);
  const dim3 grid(unsigned(row_tiles), unsigned(min64(col_tiles, 65535)));
  transpose_kernel<S, D><<<grid, kThreads, 0, as_stream(stream)>>>(
      static_cast<const S*>(src), rows, cols, src_ld, static_cast<D*>(dst), dst_ld, col_tiles);
  PARRM_LAUNCH_OK("parrm_transpose");
  return PARRM_OK;
}

// destination: float64, float32 or (checked by the caller) the source type itself
template <typename S>
int dispatch_dst(const void* src, int64_t rows, int64_t cols, int64_t src_ld,
                 void* dst, int dst_type, int64_t dst_ld, void* stream) {
  if (dst_type == PARRM_F64) return launch<S, double>(src, rows, cols, src_ld, dst, dst_ld, stream);
  if (dst_type == PARRM_F32) return launch<S, float>(src, rows, cols, src_ld, dst, dst_ld, stream);
  return launch<S, S>(src, rows, cols, src_ld, dst, dst_ld, stream);  // dst_type == src_type
}

}  // namespace
}  // namespace parrm

extern "C" int parrm_transpose(const void* d_src, int src_type, int64_t rows, int64_t cols,
                               int64_t src_ld, void* d_dst, int dst_type, int64_t dst_ld,
                               void* stream) {
  PARRM_REQUIRE(src_type >= PARRM_F64 && src_type <= PARRM_I32,
                "parrm_transpose: unknown source type %d", src_type);
  PARRM_REQUIRE(dst_type >= PARRM_F64 && dst_type <= PARRM_I32,
                "parrm_transpose: unknown destination type %d", dst_type);
  PARRM_REQUIRE(dst_type == src_type || dst_type == PARRM_F64 || dst_type == PARRM_F32,
                "parrm_transpose: unsupported type pair %d -> %d (the destination is the source "
                "type, float64 or float32)", src_type, dst_type);
  PARRM_REQUIRE(rows >= 0 && cols >= 0, "parrm_transpose: negative shape %lld x %lld",
                (long long)rows, (long long)cols);
  PARRM_REQUIRE(src_ld >= cols, "parrm_transpose: src_ld %lld < cols %lld",
                (long long)src_ld, (long long)cols);
  PARRM_REQUIRE(dst_ld >= rows, "parrm_transpose: dst_ld %lld < rows %lld",
                (long long)dst_ld, (long long)rows);
  PARRM_REQUIRE(d_src != nullptr && d_dst != nullptr, "parrm_transpose: null pointer");
  if (rows == 0 || cols == 0) return PARRM_OK;
  using namespace parrm;
  switch (src_type) {
    case PARRM_F64: return dispatch_dst<double>(d_src, rows, cols, src_ld, d_dst, dst_type, dst_ld, stream);
    case PARRM_F32: return dispatch_dst<float>(d_src, rows, cols, src_ld, d_dst, dst_type, dst_ld, stream);
    case PARRM_I16: return dispatch_dst<int16_t>(d_src, rows, cols, src_ld, d_dst, dst_type, dst_ld, stream);
    default: return dispatch_dst<int32_t>(d_src, rows, cols, src_ld, d_dst, dst_type, dst_ld, stream);
  }
}
