// Period filter: body of PARRM.filter_data (parrm.py:861-869) as a direct gather.
//
//   y[c,t] = x[c,t] - (1/n_in(t)) * sum_{w in taps, 0 <= t-w < T} x[c,t-w];   0 where n_in(t) = 0
//
// The reference evaluates this with two FFT convolutions (the second one, of an all-ones
// array, only counts the in-range taps).  Here every CTA stages one time tile plus its halo
// [t0 - w_max, t0 + tile - w_min) of one channel into shared memory with a single TMA bulk
// copy (cp.async.bulk, SASS UBLKCP) and gathers the taps from there.  HBM traffic is the
// algorithmic 2 * sizeof(T) bytes per channel-sample; the halo re-reads of neighbouring
// tiles are served by L2.
#include <string.h>

#include "common.cuh"
#include "filter_jit.h"
#include "filter_plan.h"
#include "gather.cuh"

namespace parrm {

// name of the kernel the last parrm_filter_apply* call of this thread enqueued
static thread_local const char* g_last_kernel = "";

template <typename T>
struct FilterArgs {
  const T* x;
  T* out;
  const int32_t* taps;  // device, ascending
  int64_t ld_x, x_t0, n_x;
  int64_t ld_out, t0, n_out;
  int64_t n_total;
  int32_t n_taps, w_lo, w_hi;  // w_lo = min(w_min, 0), w_hi = max(w_max, 0)
  int32_t tile;
};

// ---- shared-memory gather --------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kGatherThreads)
filter_gather_smem_kernel(const FilterArgs<T> a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
  int32_t* s_taps = reinterpret_cast<int32_t*>(smem_raw + 16);
  T* s_win = reinterpret_cast<T*>(smem_raw + 16 + round16(a.n_taps * 4));
  constexpr int VEC = 16 / sizeof(T);

  const int tid = threadIdx.x;
  const int64_t chan = blockIdx.y;
  const int64_t tile_t0 = a.t0 + int64_t(blockIdx.x) * a.tile;
  const int n_tile = int(min(int64_t(a.tile), a.t0 + a.n_out - tile_t0));
  // window of global sample times held in shared memory
  const int64_t g_lo = tile_t0 - a.w_hi;
  const int64_t g_hi = tile_t0 + n_tile - a.w_lo;
  const int64_t v_lo = max(g_lo, max(int64_t(0), a.x_t0));
  const int64_t v_hi = min(g_hi, min(a.n_total, a.x_t0 + a.n_x));
  const T* xrow = a.x + chan * a.ld_x - a.x_t0;  // xrow[g] = sample at global time g

  // Element shift of the window so that 16-byte aligned global addresses land on 16-byte
  // aligned shared addresses (bulk-copy requirement).
  const int g_mis = int((reinterpret_cast<uintptr_t>(xrow + v_lo) / sizeof(T)) % VEC);
  const int shift = (g_mis - int((v_lo - g_lo) % VEC) + VEC) % VEC;
  T* s_x = s_win + shift;  // s_x[g - g_lo]
  const int n_valid = int(v_hi - v_lo);
  const int head = min((VEC - g_mis) % VEC, n_valid);
  const int n_bulk = ((n_valid - head) / VEC) * VEC;

  if (tid == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (tid == 0 && n_bulk > 0) {
    mbar_expect_tx(bar, uint32_t(n_bulk) * sizeof(T));
    bulk_g2s(s_x + (v_lo - g_lo) + head, xrow + v_lo + head, uint32_t(n_bulk) * sizeof(T), bar);
  }
  for (int i = tid; i < a.n_taps; i += kGatherThreads) s_taps[i] = a.taps[i];
  // scalar head / tail around the bulk copy, zero fill outside the recording
  if (tid < head) s_x[(v_lo - g_lo) + tid] = xrow[v_lo + tid];
  for (int i = head + n_bulk + tid; i < n_valid; i += kGatherThreads)
    s_x[(v_lo - g_lo) + i] = xrow[v_lo + i];
  for (int i = tid; i < int(v_lo - g_lo); i += kGatherThreads) s_x[i] = T(0);
  for (int i = int(v_hi - g_lo) + tid; i < int(g_hi - g_lo); i += kGatherThreads) s_x[i] = T(0);
  __syncthreads();
  if (n_bulk > 0) mbar_wait(bar, 0);

  T* orow = a.out + chan * a.ld_out + (tile_t0 - a.t0);
  const bool interior = (g_lo >= 0) && (g_hi <= a.n_total);
  gather_tile<T>(s_x + a.w_hi, s_taps, a.n_taps, n_tile, interior, tile_t0, a.n_total,
                 [=](int i, T y) { orow[i] = y; });
}

// ---- global-memory gather (spans or tap lists too large for shared memory) --------
template <typename T>
__global__ void __launch_bounds__(kGatherThreads)
filter_gather_global_kernel(const FilterArgs<T> a) {
  const int64_t chan = blockIdx.y;
  const T* xrow = a.x + chan * a.ld_x - a.x_t0;
  T* orow = a.out + chan * a.ld_out - a.t0;
  for (int64_t t = a.t0 + int64_t(blockIdx.x) * kGatherThreads + threadIdx.x; t < a.t0 + a.n_out;
       t += int64_t(gridDim.x) * kGatherThreads) {
    orow[t] = gather_point<T>(t, a.taps, a.n_taps, a.n_total,
                              [=](int64_t src) { return xrow[src]; });
  }
}

// ---- batched gather: many tap sets over the same recording in ONE launch ------------
// The parameter explorer (and any parameter sweep) filters one short recording with many
// (half-width, period half-width, omit, direction) sets.  blockIdx.z is the set; its taps and
// tap count are read from device memory (straight from parrm_build_taps_batch, no host round
// trip); the staged window is sized for the widest set.  Every output counts its in-range
// taps (the edge form of gather_tile): this path is for small data, not for throughput.
template <typename T>
__global__ void __launch_bounds__(kGatherThreads)
filter_gather_batch_kernel(const T* __restrict__ x, int64_t ld_x, int64_t n_total,
                           const int32_t* __restrict__ taps, int64_t tap_stride,
                           const int32_t* __restrict__ n_taps_of, int32_t w_max, int32_t tile,
                           T* __restrict__ out, int64_t ld_out, int64_t set_stride) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  T* const s_win = reinterpret_cast<T*>(smem_raw);                    // [tile + 2 w_max]
  int32_t* const s_taps = reinterpret_cast<int32_t*>(s_win + tile + 2 * w_max);
  const int64_t set = blockIdx.z, chan = blockIdx.y;
  const int64_t t_lo = int64_t(blockIdx.x) * tile;
  const int n_tile = int(min64(tile, n_total - t_lo));
  const int n_taps = n_taps_of[set];
  const T* const row = x + chan * ld_x;
  for (int i = threadIdx.x; i < n_tile + 2 * w_max; i += kGatherThreads) {
    const int64_t g = t_lo - w_max + i;
    s_win[i] = (g >= 0 && g < n_total) ? row[g] : T(0);
  }
  for (int i = threadIdx.x; i < n_taps; i += kGatherThreads) s_taps[i] = taps[set * tap_stride + i];
  __syncthreads();
  T* const orow = out + set * set_stride + chan * ld_out + t_lo;
  gather_tile<T>(s_win + w_max, s_taps, n_taps, n_tile, false, t_lo, n_total,
                 [=](int i, T y) { orow[i] = y; });
}

template <typename T>
int launch_filter(const FilterArgs<T>& args_in, int64_t n_chans, cudaStream_t stream) {
  FilterArgs<T> a = args_in;
  const int64_t span = int64_t(a.w_hi) - a.w_lo;
  const int64_t fixed = 16 + round16(a.n_taps * 4) + 32;
  const int64_t min_window = (1024 + span) * int64_t(sizeof(T));
  if (fixed + min_window > kGatherSmemBudget) {
    const int64_t blocks = min64(ceil_div(a.n_out, kGatherThreads), 148 * 32);
    dim3 grid((unsigned)blocks, (unsigned)n_chans);
    filter_gather_global_kernel<T><<<grid, kGatherThreads, 0, stream>>>(a);
    PARRM_LAUNCH_OK("filter_gather_global_kernel");
    g_last_kernel = "filter_gather_global_kernel";
    return PARRM_OK;
  }
  // tile: at least the halo span (<= 2x read amplification from L2), in 1024-output passes
  int64_t tile = ((span + 1023) / 1024) * 1024;
  tile = max64(4096, min64(tile, 8192));
  while (fixed + (tile + span) * int64_t(sizeof(T)) > kGatherSmemBudget) tile -= 1024;
  tile = min64(tile, ((a.n_out + 1023) / 1024) * 1024);
  a.tile = int32_t(tile);
  const size_t smem = size_t(fixed + (tile + span + 16 / sizeof(T)) * sizeof(T));
  PARRM_CUDA_OK(cudaFuncSetAttribute(filter_gather_smem_kernel<T>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  dim3 grid((unsigned)ceil_div(a.n_out, tile), (unsigned)n_chans);
  filter_gather_smem_kernel<T><<<grid, kGatherThreads, smem, stream>>>(a);
  PARRM_LAUNCH_OK("filter_gather_smem_kernel");
  g_last_kernel = "filter_gather_smem_kernel";
  return PARRM_OK;
}


}  // namespace parrm

extern "C" {

const char* parrm_filter_last_kernel(void) { return parrm::g_last_kernel; }

int parrm_filter_specialise_check(const void* h_plan, int dtype,
                                  const parrm_filter_options_t* options, int32_t* shape,
                                  size_t* cubin_bytes) {
  using namespace parrm;
  PARRM_REQUIRE(h_plan != nullptr, "parrm_filter_specialise_check: null plan");
  const FilterPlanHeader* hdr = static_cast<const FilterPlanHeader*>(h_plan);
  PARRM_REQUIRE(hdr->magic == kPlanMagic && hdr->version == kPlanVersion,
                "parrm_filter_specialise_check: not a filter plan");
  const int32_t* h_terms = reinterpret_cast<const int32_t*>(
      static_cast<const unsigned char*>(h_plan) + hdr->terms_offset);
  FilterTuning tune{0, options ? options->steps_per_chunk : 0,
                    options ? options->prefetch_chunks : 0, options ? options->ctas_per_sm : 0,
                    options ? options->variant : 0, options ? options->timeline : 0};
  CombEShape s;
  if (!comb_e_shape(hdr, h_terms, dtype, &tune, &s)) {
    set_error("parrm_filter_specialise_check: this plan is outside the specialised kernel's range");
    return PARRM_ERR_UNSUPPORTED;
  }
  if (shape) {
    const int32_t v[12] = {s.d, s.nk, s.m[0], s.m[1], s.nb[0], s.nb[1], s.n_plus + s.n_minus,
                           s.u, s.pf, s.ctas, s.smem_bytes, ((s.d + 31) / 32) * 32 + 32};
    for (int i = 0; i < 12; ++i) shape[i] = v[i];
  }
  if (cubin_bytes == nullptr) return PARRM_OK;  // range check only
  return comb_e_compile_only(s, cubin_bytes);
}

int parrm_filter_apply(const void* d_x, int64_t ld_x, int64_t x_t0, int64_t n_x, void* d_out,
                       int64_t ld_out, int64_t t0, int64_t n_out, int64_t n_samples_total,
                       int64_t n_chans, const void* d_plan, const void* h_plan, int dtype,
                       void* stream) {
  return parrm_filter_apply_ex(d_x, ld_x, x_t0, n_x, d_out, ld_out, t0, n_out, n_samples_total,
                               n_chans, d_plan, h_plan, dtype, nullptr, stream);
}

int parrm_filter_apply_ex(const void* d_x, int64_t ld_x, int64_t x_t0, int64_t n_x, void* d_out,
                          int64_t ld_out, int64_t t0, int64_t n_out, int64_t n_samples_total,
                          int64_t n_chans, const void* d_plan, const void* h_plan, int dtype,
                          const parrm_filter_options_t* options, void* stream) {
  PARRM_NVTX("parrm_filter_apply_ex");
  using namespace parrm;
  PARRM_REQUIRE(d_plan != nullptr && h_plan != nullptr, "parrm_filter_apply: null plan");
  const FilterPlanHeader* hdr = static_cast<const FilterPlanHeader*>(h_plan);
  PARRM_REQUIRE(hdr->magic == kPlanMagic && hdr->version == kPlanVersion,
                "parrm_filter_apply: not a filter plan");
  PARRM_REQUIRE(hdr->dtype == dtype, "parrm_filter_apply: plan built for another dtype");
  PARRM_REQUIRE(dtype == PARRM_F64 || dtype == PARRM_F32, "parrm_filter_apply: bad dtype %d", dtype);
  PARRM_REQUIRE(n_chans >= 0 && n_out >= 0 && n_x >= 0 && n_samples_total >= 0,
                "parrm_filter_apply: negative size");
  PARRM_REQUIRE(n_chans <= 65535, "parrm_filter_apply: more than 65535 channels per call");
  const int want = options ? options->kernel : PARRM_FILTER_KERNEL_AUTO;
  PARRM_REQUIRE(want == PARRM_FILTER_KERNEL_AUTO || want == PARRM_FILTER_KERNEL_GATHER ||
                    want == PARRM_FILTER_KERNEL_SPECIALISED,
                "parrm_filter_apply: unknown kernel choice %d", want);
  if (n_chans == 0 || n_out == 0) return PARRM_OK;
  PARRM_REQUIRE(d_x != nullptr && d_out != nullptr, "parrm_filter_apply: null data pointer");
  PARRM_REQUIRE(t0 >= 0 && t0 + n_out <= n_samples_total,
                "parrm_filter_apply: output range outside the recording");
  const int32_t w_lo = hdr->w_min < 0 ? hdr->w_min : 0;
  const int32_t w_hi = hdr->w_max > 0 ? hdr->w_max : 0;
  {
    const int64_t need_lo = t0 - w_hi > 0 ? t0 - w_hi : 0;
    const int64_t need_hi =
        t0 + n_out - w_lo < n_samples_total ? t0 + n_out - w_lo : n_samples_total;
    PARRM_REQUIRE(x_t0 <= need_lo && x_t0 + n_x >= need_hi,
                  "parrm_filter_apply: input chunk [%lld, %lld) does not cover the halo [%lld, %lld)",
                  (long long)x_t0, (long long)(x_t0 + n_x), (long long)need_lo, (long long)need_hi);
  }
  const unsigned char* h_base = static_cast<const unsigned char*>(h_plan);
  const int32_t* d_taps = reinterpret_cast<const int32_t*>(
      static_cast<const unsigned char*>(d_plan) + hdr->taps_offset);
  const int32_t* h_terms = reinterpret_cast<const int32_t*>(h_base + hdr->terms_offset);
  cudaStream_t s = as_stream(stream);

  // 1. kernel specialised for this plan at run time (pattern-first comb, filter_comb_e.cuh).
  //    Building it costs about a second once per plan, so short one-off calls keep the
  //    pre-built gather unless the specialisation already exists.
  if (hdr->kind == kPlanComb &&
      (want == PARRM_FILTER_KERNEL_AUTO || want == PARRM_FILTER_KERNEL_SPECIALISED)) {
    FilterTuning tune{want, options ? options->steps_per_chunk : 0,
                      options ? options->prefetch_chunks : 0, options ? options->ctas_per_sm : 0,
                    options ? options->variant : 0, options ? options->timeline : 0};
    CombEShape shape;
    const bool fits = comb_e_shape(hdr, h_terms, dtype, &tune, &shape);
    const bool worth = want == PARRM_FILTER_KERNEL_SPECIALISED ||
                       n_chans * n_out >= (int64_t(1) << 24) || (fits && comb_e_cached(shape));
    if (fits && worth) {
      const unsigned char* d_base = static_cast<const unsigned char*>(d_plan);
      const int rc = launch_comb_e(
          shape, d_x, d_out, d_taps,
          reinterpret_cast<const int32_t*>(d_base + hdr->count_offset),
          reinterpret_cast<const double*>(d_base + hdr->recip_offset), ld_x, x_t0, n_x, ld_out,
          t0, n_out, n_samples_total, n_chans, s, nullptr, tune.timeline);
      if (rc == PARRM_OK) {
        g_last_kernel = "parrm_filter_comb_e";
        return rc;
      }
      if (rc != PARRM_ERR_UNSUPPORTED || want == PARRM_FILTER_KERNEL_SPECIALISED) return rc;
    } else if (want == PARRM_FILTER_KERNEL_SPECIALISED) {
      set_error("parrm_filter_apply: this plan is outside the specialised kernel's range");
      return PARRM_ERR_UNSUPPORTED;
    }
  } else if (want == PARRM_FILTER_KERNEL_SPECIALISED) {
    set_error("parrm_filter_apply: the specialised kernel needs a comb plan");
    return PARRM_ERR_UNSUPPORTED;
  }

  // 2. pre-built gather: one shared-memory load per tap (any tap set, any size)
  if (dtype == PARRM_F64) {
    FilterArgs<double> a{static_cast<const double*>(d_x), static_cast<double*>(d_out),
                         d_taps, ld_x, x_t0, n_x, ld_out, t0, n_out, n_samples_total,
                         hdr->n_taps, w_lo, w_hi, 0};
    return launch_filter<double>(a, n_chans, s);
  }
  FilterArgs<float> a{static_cast<const float*>(d_x), static_cast<float*>(d_out),
                      d_taps, ld_x, x_t0, n_x, ld_out, t0, n_out, n_samples_total,
                      hdr->n_taps, w_lo, w_hi, 0};
  return launch_filter<float>(a, n_chans, s);
}

int parrm_filter_apply_batch(const void* d_x, int64_t ld_x, int64_t n_samples, int64_t n_chans,
                             const int32_t* d_taps, int64_t tap_stride, const int32_t* d_n_taps,
                             int64_t n_sets, int64_t max_half_width, void* d_out, int64_t ld_out,
                             int64_t set_stride, int dtype, void* stream) {
  PARRM_NVTX("parrm_filter_apply_batch");
  using namespace parrm;
  PARRM_REQUIRE(dtype == PARRM_F64 || dtype == PARRM_F32, "parrm_filter_apply_batch: bad dtype %d", dtype);
  PARRM_REQUIRE(n_sets >= 0 && n_sets <= 65535 && n_chans >= 0 && n_chans <= 65535 && n_samples >= 0,
                "parrm_filter_apply_batch: bad shape");
  if (n_sets == 0 || n_chans == 0 || n_samples == 0) return PARRM_OK;
  PARRM_REQUIRE(d_x && d_taps && d_n_taps && d_out, "parrm_filter_apply_batch: null pointer");
  const size_t es = dtype == PARRM_F64 ? 8 : 4;
  PARRM_REQUIRE(max_half_width >= 1 && tap_stride >= 1, "parrm_filter_apply_batch: empty tap rows");
  const int64_t tile = 2048;
  const size_t smem = size_t(tile + 2 * max_half_width) * es + size_t(tap_stride) * 4;
  PARRM_REQUIRE(smem <= size_t(kGatherSmemBudget),
                "parrm_filter_apply_batch: half-width %lld too wide for the batched kernel "
                "(filter the sets one by one with parrm_filter_apply)", (long long)max_half_width);
  dim3 grid(unsigned(ceil_div(n_samples, tile)), unsigned(n_chans), unsigned(n_sets));
  if (dtype == PARRM_F64) {
    auto kernel = filter_gather_batch_kernel<double>;
    PARRM_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    kernel<<<grid, kGatherThreads, smem, as_stream(stream)>>>(
        static_cast<const double*>(d_x), ld_x, n_samples, d_taps, tap_stride, d_n_taps,
        int32_t(max_half_width), int32_t(tile), static_cast<double*>(d_out), ld_out, set_stride);
  } else {
    auto kernel = filter_gather_batch_kernel<float>;
    PARRM_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    kernel<<<grid, kGatherThreads, smem, as_stream(stream)>>>(
        static_cast<const float*>(d_x), ld_x, n_samples, d_taps, tap_stride, d_n_taps,
        int32_t(max_half_width), int32_t(tile), static_cast<float*>(d_out), ld_out, set_stride);
  }
  PARRM_LAUNCH_OK("filter_gather_batch_kernel");
  g_last_kernel = "filter_gather_batch_kernel";
  return PARRM_OK;
}

}  // extern "C"
