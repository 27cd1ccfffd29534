// Gather arithmetic of the period filter, shared by the whole-recording kernels (filter.cu) and
// the streaming kernels (stream.cu):
//
//   y[t] = x[t] - (1/n_in(t)) * sum_{w in taps, 0 <= t-w < n_total} x[t-w];   0 where n_in(t) = 0
//
// Every gather output of the library is computed by gather_tile or gather_point below, so the
// operations and their order are fixed in one place: ascending taps, sequential adds,
// acc / n_taps in the interior, acc / n_in at the edges, finite_or_zero(x - mean).  That is what
// makes a streamed recording bit-equal to filter_data with a gather plan on the whole of it.
// The callers differ only in where samples come from and where outputs go, which they pass in
// as a load or store lambda.  The lambdas capture by value: with a by-reference capture nvcc
// 12.9 unrolls the float tap loop of filter_gather_global_kernel differently.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace parrm {

constexpr int kGatherThreads = 256;     // threads per CTA of every gather kernel
constexpr int kGatherOutPerThread = 4;  // outputs per thread and pass of the interior form
constexpr int kGatherSmemBudget = 200 * 1024;

__host__ __device__ inline int round16(int bytes) { return (bytes + 15) & ~15; }

// parrm.py:869: outputs that are not finite become 0 (a NaN/Inf sample zeroes exactly the
// outputs whose tap window, or own sample, contains it)
template <typename T>
__device__ __forceinline__ T finite_or_zero(T y) {
  return isfinite(y) ? y : T(0);
}

// Outputs [tile_t0, tile_t0 + n_tile) from a staged window, s_c[i] = sample tile_t0 + i, with
// s_taps the ascending taps in shared memory; store(i, y) writes output tile_t0 + i.  interior:
// every tap of every output lies in [0, n_total), so each output divides by n_taps; otherwise each
// output counts its in-range taps and reads only those.  Called by all threads of the CTA.
template <typename T, typename Store>
__device__ __forceinline__ void gather_tile(const T* s_c, const int32_t* s_taps, int n_taps,
                                            int n_tile, bool interior, int64_t tile_t0,
                                            int64_t n_total, Store store) {
  const int tid = threadIdx.x;
  if (interior) {
    const T inv_scale = T(n_taps);
    for (int i0 = tid; i0 < n_tile; i0 += kGatherThreads * kGatherOutPerThread) {
      T acc[kGatherOutPerThread];
#pragma unroll
      for (int r = 0; r < kGatherOutPerThread; ++r) acc[r] = T(0);
      // clamp the per-thread outputs of a ragged last pass onto a valid one
      int idx[kGatherOutPerThread];
#pragma unroll
      for (int r = 0; r < kGatherOutPerThread; ++r)
        idx[r] = min(i0 + r * kGatherThreads, n_tile - 1);
#pragma unroll 4
      for (int k = 0; k < n_taps; ++k) {
        const int w = s_taps[k];
#pragma unroll
        for (int r = 0; r < kGatherOutPerThread; ++r) acc[r] += s_c[idx[r] - w];
      }
#pragma unroll
      for (int r = 0; r < kGatherOutPerThread; ++r) {
        const int i = i0 + r * kGatherThreads;
        if (i < n_tile) store(i, finite_or_zero(s_c[i] - acc[r] / inv_scale));
      }
    }
  } else {
    for (int i = tid; i < n_tile; i += kGatherThreads) {
      const int64_t t = tile_t0 + i;
      T acc = T(0);
      int n_in = 0;
      for (int k = 0; k < n_taps; ++k) {
        const int w = s_taps[k];
        const int64_t src = t - w;
        if (src >= 0 && src < n_total) {
          acc += s_c[i - w];
          ++n_in;
        }
      }
      store(i, n_in > 0 ? finite_or_zero(s_c[i] - acc / T(n_in)) : T(0));
    }
  }
}

// Output t read straight from memory, for tap windows too wide to stage: load(s) returns sample
// s, and only samples in [0, n_total) are loaded.
template <typename T, typename Load>
__device__ __forceinline__ T gather_point(int64_t t, const int32_t* taps, int n_taps,
                                          int64_t n_total, Load load) {
  T acc = T(0);
  int n_in = 0;
  for (int k = 0; k < n_taps; ++k) {
    const int64_t src = t - taps[k];
    if (src >= 0 && src < n_total) {
      acc += load(src);
      ++n_in;
    }
  }
  return n_in > 0 ? finite_or_zero(load(t) - acc / T(n_in)) : T(0);
}

}  // namespace parrm
