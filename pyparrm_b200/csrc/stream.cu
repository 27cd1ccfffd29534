// Streaming filter: filter_data applied block by block as a recording is acquired.
//
// State per stream (all caller-owned device memory):
//   ring[c * R + (t mod R)]  the last R samples of every channel, in the compute type, with
//                            R = span + max_chunk,  span = max(w_max, 0) - min(w_min, 0);
//   taps                     ascending offsets, as parrm_build_taps produces them;
//   pos, out_lo              samples pushed before this block and the first output not yet
//                            written (host arguments, or a device int64 header so that a
//                            captured CUDA graph can replay with new positions).
//
// One launch per push.  The block holds samples [pos, pos + n) in its storage type.  Output t
// reads samples t - w for the taps w; it is final once sample t + L exists, L = max(0, -w_min),
// so while the stream is open a push produces outputs [out_lo, max(out_lo, pos + n - L)) and the
// closing push the rest, up to pos + n, with the recording-end edge.  Treating the recording as
// ending at pos + n is exact for the open outputs too: none of their taps reaches past it.  With
// one tap set for the whole stream out_lo = max(0, pos - L) (parrm_stream_push); after a switch
// of taps the caller passes it (parrm_stream_push_at), and a push can then emit more or fewer
// than n outputs.
//
// Every CTA reads samples >= pos from the incoming block and older ones from the ring, and
// writes only its own slice of the block into the ring.  The oldest sample any output of this
// launch reads is out_lo - w_max, and the caller guarantees R >= pos + n - that (R >= span + n
// for a single tap set), so the slots written here ((pos .. pos+n-1) mod R) are never slots read
// here: no grid-wide barrier is needed.  Work and traffic per push are O(channels x (n + span +
// pos - out_lo)), independent of how much has been pushed.
//
// Arithmetic: both kernels compute their outputs with the gather body of gather.cuh, the same
// gather_tile / gather_point that the gather kernels of filter.cu call, so a streamed recording
// is bit-equal to filter_data with a gather plan on the whole of it by construction.  Only the
// staging differs (ring + block here).  Widening from the storage type is parrm_convert's
// static_cast, narrowing to the output type likewise.
#include <limits.h>

#include "common.cuh"
#include "gather.cuh"

namespace parrm {

template <typename T>
struct StreamArgs {
  T* ring;
  const int32_t* taps;
  const void* block;
  void* out;
  const int64_t* d_hdr;  // {pos} (hdr_words 1) or {pos, out_lo} (hdr_words 2), or NULL
  int64_t ring_len, ld_block, n, ld_out, pos, out_lo;
  int32_t n_taps, w_lo, w_hi, tile;
  int32_t block_type, out_type, close, hdr_words;
};

template <typename T>
__device__ __forceinline__ T load_block(const void* b, int type, int64_t i) {
  switch (type) {
    case PARRM_F64: return static_cast<T>(static_cast<const double*>(b)[i]);
    case PARRM_F32: return static_cast<T>(static_cast<const float*>(b)[i]);
    case PARRM_I16: return static_cast<T>(static_cast<const int16_t*>(b)[i]);
    default: return static_cast<T>(static_cast<const int32_t*>(b)[i]);
  }
}

template <typename T>
__device__ __forceinline__ void store_out(void* o, int type, int64_t i, T y) {
  if (type == PARRM_F64)
    static_cast<double*>(o)[i] = static_cast<double>(y);
  else
    static_cast<float*>(o)[i] = static_cast<float>(y);
}

// Latency L = max(0, -w_min) of a tap set, and the end of the outputs a push of samples up to
// `end` makes final: all of them when the stream closes, else those up to end - L.
__host__ __device__ inline int64_t stream_latency(int32_t w_min) {
  return w_min < 0 ? -int64_t(w_min) : 0;
}
__host__ __device__ inline int64_t stream_out_hi(int64_t end, int64_t out_lo, int64_t lat,
                                                 int close) {
  return close ? end : (end - lat > out_lo ? end - lat : out_lo);
}

// Position, output range and recording end of this push (identical in every CTA).
struct StreamRange {
  int64_t pos, out_lo, out_hi, n_total;
};

template <typename T>
__device__ __forceinline__ StreamRange stream_range(const StreamArgs<T>& a) {
  StreamRange r;
  const int64_t lat = stream_latency(a.w_lo);
  if (a.d_hdr == nullptr) {
    r.pos = a.pos;
    r.out_lo = a.out_lo;
  } else {
    r.pos = a.d_hdr[0];
    r.out_lo = a.hdr_words == 2 ? a.d_hdr[1] : max(int64_t(0), r.pos - lat);
  }
  r.n_total = r.pos + a.n;
  r.out_hi = stream_out_hi(r.n_total, r.out_lo, lat, a.close);
  return r;
}

// This CTA's slice [x * tile, (x + 1) * tile) of the block, widened, into the ring.
template <typename T>
__device__ __forceinline__ void block_to_ring(const StreamArgs<T>& a, const StreamRange& r,
                                              int64_t chan) {
  const int64_t b0 = int64_t(blockIdx.x) * a.tile;
  const int64_t b1 = min(b0 + a.tile, a.n);
  if (b0 >= b1) return;
  T* ring = a.ring + chan * a.ring_len;
  const int64_t base = (r.pos + b0) % a.ring_len;  // the slice is shorter than R: one wrap at most
  for (int64_t i = b0 + threadIdx.x; i < b1; i += kGatherThreads) {
    int64_t j = base + (i - b0);
    if (j >= a.ring_len) j -= a.ring_len;
    ring[j] = load_block<T>(a.block, a.block_type, chan * a.ld_block + i);
  }
}

// ---- shared-memory gather: one output tile + its tap window per CTA ------------------------
template <typename T>
__global__ void __launch_bounds__(kGatherThreads)
stream_gather_smem_kernel(const StreamArgs<T> a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int32_t* s_taps = reinterpret_cast<int32_t*>(smem_raw);
  T* s_win = reinterpret_cast<T*>(smem_raw + round16(a.n_taps * 4));
  const int tid = threadIdx.x;
  const int64_t chan = blockIdx.y;
  const StreamRange r = stream_range(a);
  block_to_ring(a, r, chan);

  const int64_t tile_t0 = r.out_lo + int64_t(blockIdx.x) * a.tile;
  if (tile_t0 >= r.out_hi) return;
  const int n_tile = int(min(int64_t(a.tile), r.out_hi - tile_t0));
  const int64_t g_lo = tile_t0 - a.w_hi;              // window of sample times in s_win
  const int64_t g_hi = tile_t0 + n_tile - a.w_lo;
  const int64_t v_lo = max(g_lo, int64_t(0));
  const int64_t v_mid = max(v_lo, min(g_hi, r.pos));  // [v_lo, v_mid) from the ring
  const int64_t v_hi = min(g_hi, r.n_total);          // [v_mid, v_hi) from the block
  const T* ring = a.ring + chan * a.ring_len;
  const int64_t ring0 = v_lo % a.ring_len;            // fewer than R samples: one wrap at most

  for (int i = tid; i < a.n_taps; i += kGatherThreads) s_taps[i] = a.taps[i];
  for (int i = tid; i < int(g_hi - g_lo); i += kGatherThreads) {
    const int64_t g = g_lo + i;
    T v = T(0);
    if (g >= v_lo && g < v_mid) {
      int64_t j = ring0 + (g - v_lo);
      if (j >= a.ring_len) j -= a.ring_len;
      v = ring[j];
    } else if (g >= v_mid && g < v_hi) {
      v = load_block<T>(a.block, a.block_type, chan * a.ld_block + (g - r.pos));
    }
    s_win[i] = v;
  }
  __syncthreads();

  const int64_t o0 = chan * a.ld_out + (tile_t0 - r.out_lo);
  const bool interior = (g_lo >= 0) && (g_hi <= r.n_total);
  gather_tile<T>(s_win + a.w_hi, s_taps, a.n_taps, n_tile, interior, tile_t0, r.n_total,
                 [=](int i, T y) { store_out(a.out, a.out_type, o0 + i, y); });
}

// ---- global-memory gather: tap windows too wide for shared memory -------------------------
// The ring of such a stream is read from L2 (384 channels x a 4 k-sample span x 8 B ~ 12 MB).
template <typename T>
__global__ void __launch_bounds__(kGatherThreads)
stream_gather_global_kernel(const StreamArgs<T> a) {
  const int64_t chan = blockIdx.y;
  const StreamRange r = stream_range(a);
  block_to_ring(a, r, chan);
  const int64_t t = r.out_lo + int64_t(blockIdx.x) * a.tile + threadIdx.x;
  if (t >= r.out_hi) return;
  const T* ring = a.ring + chan * a.ring_len;
  const int64_t blk = chan * a.ld_block - r.pos;  // block element of sample s >= pos: blk + s
  const T y = gather_point<T>(t, a.taps, a.n_taps, r.n_total, [=](int64_t s) {
    return s >= r.pos ? load_block<T>(a.block, a.block_type, blk + s) : ring[s % a.ring_len];
  });
  store_out(a.out, a.out_type, chan * a.ld_out + (t - r.out_lo), y);
}

static int64_t stream_span(int32_t w_min, int32_t w_max) {
  return int64_t(w_max > 0 ? w_max : 0) - int64_t(w_min < 0 ? w_min : 0);
}

template <typename T>
int launch_stream(StreamArgs<T> a, int64_t n_chans, int64_t n_out_max, cudaStream_t stream) {
  // n_out_max covers both the outputs and the block: CTA x also writes block slice x to the ring
  const int64_t span = int64_t(a.w_hi) - a.w_lo;
  const int64_t fixed = round16(a.n_taps * 4);
  const int64_t es = int64_t(sizeof(T));
  if (fixed + (kGatherThreads + span) * es > kGatherSmemBudget) {
    a.tile = kGatherThreads;
    dim3 grid(unsigned(ceil_div(n_out_max, a.tile)), unsigned(n_chans));
    stream_gather_global_kernel<T><<<grid, kGatherThreads, 0, stream>>>(a);
    PARRM_LAUNCH_OK("stream_gather_global_kernel");
    return PARRM_OK;
  }
  // Tiles of 256..4096 outputs: enough CTAs to cover the GPU twice when the push allows it,
  // no more outputs per CTA than the push has, and the window within the shared-memory budget.
  const int64_t want = ceil_div(n_out_max * n_chans, 2 * int64_t(kNumSMs));
  int64_t tile = ceil_div(max64(want, 1), kGatherThreads) * kGatherThreads;
  tile = min64(min64(tile, 4096), ceil_div(n_out_max, kGatherThreads) * kGatherThreads);
  while (tile > kGatherThreads && fixed + (tile + span) * es > kGatherSmemBudget)
    tile -= kGatherThreads;
  a.tile = int32_t(tile);
  const size_t smem = size_t(fixed + (tile + span) * es);
  PARRM_CUDA_OK(cudaFuncSetAttribute(stream_gather_smem_kernel<T>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  dim3 grid(unsigned(ceil_div(n_out_max, tile)), unsigned(n_chans));
  stream_gather_smem_kernel<T><<<grid, kGatherThreads, smem, stream>>>(a);
  PARRM_LAUNCH_OK("stream_gather_smem_kernel");
  return PARRM_OK;
}

}  // namespace parrm

extern "C" {

size_t parrm_stream_ring_bytes(int64_t n_chans, const int32_t* h_taps, int32_t n_taps,
                               int64_t max_chunk, int dtype) {
  using namespace parrm;
  if (h_taps == nullptr || n_taps < 1 || n_chans < 1 || max_chunk < 1 ||
      (dtype != PARRM_F64 && dtype != PARRM_F32)) {
    set_error("parrm_stream_ring_bytes: need taps, channels >= 1, max_chunk >= 1 and a "
              "float64 / float32 compute type");
    return 0;
  }
  for (int32_t i = 1; i < n_taps; ++i) {
    if (h_taps[i] <= h_taps[i - 1]) {
      set_error("parrm_stream_ring_bytes: taps must be strictly ascending");
      return 0;
    }
  }
  const int64_t ring_len = stream_span(h_taps[0], h_taps[n_taps - 1]) + max_chunk;
  return size_t(n_chans) * size_t(ring_len) * (dtype == PARRM_F64 ? 8 : 4);
}

// The body of both push entry points: arguments already checked except those below.
static int stream_push_impl(const char* fn, void* d_ring, int64_t ring_len, int64_t n_chans,
                            const int32_t* d_taps, int32_t n_taps, int32_t w_min, int32_t w_max,
                            const void* d_block, int block_type, int64_t ld_block, int64_t n,
                            void* d_out, int out_type, int64_t ld_out, int64_t pos,
                            int64_t out_lo, int64_t n_grid, const int64_t* d_hdr, int hdr_words,
                            int close, int dtype, void* stream) {
  using namespace parrm;
  PARRM_REQUIRE(dtype == PARRM_F64 || dtype == PARRM_F32, "%s: bad dtype %d", fn, dtype);
  PARRM_REQUIRE(out_type == PARRM_F64 || out_type == PARRM_F32, "%s: bad output type %d", fn,
                out_type);
  PARRM_REQUIRE(block_type == PARRM_F64 || block_type == PARRM_F32 || block_type == PARRM_I16 ||
                    block_type == PARRM_I32,
                "%s: unknown block storage type %d", fn, block_type);
  PARRM_REQUIRE(n_chans >= 1 && n_chans <= 65535, "%s: 1..65535 channels, got %lld", fn,
                (long long)n_chans);
  PARRM_REQUIRE(n_taps >= 1 && w_min <= w_max, "%s: empty or unordered tap list", fn);
  PARRM_REQUIRE(d_ring != nullptr && d_taps != nullptr, "%s: null ring or taps", fn);
  const int64_t out_hi = stream_out_hi(pos + n, out_lo, stream_latency(w_min), close);
  if (n == 0 && out_hi == out_lo) return PARRM_OK;
  PARRM_REQUIRE(n == 0 || (d_block != nullptr && ld_block >= n),
                "%s: null block or row stride %lld < %lld", fn, (long long)ld_block,
                (long long)n);
  PARRM_REQUIRE(out_hi == out_lo || (d_out != nullptr && ld_out >= out_hi - out_lo),
                "%s: null output or row stride %lld < %lld outputs", fn, (long long)ld_out,
                (long long)(out_hi - out_lo));
  const int32_t w_lo = w_min < 0 ? w_min : 0, w_hi = w_max > 0 ? w_max : 0;
  cudaStream_t s = as_stream(stream);
  if (dtype == PARRM_F64) {
    StreamArgs<double> a{static_cast<double*>(d_ring), d_taps, d_block, d_out, d_hdr, ring_len,
                         ld_block, n, ld_out, pos, out_lo, n_taps, w_lo, w_hi, 0, block_type,
                         out_type, close ? 1 : 0, hdr_words};
    return launch_stream<double>(a, n_chans, n_grid, s);
  }
  StreamArgs<float> a{static_cast<float*>(d_ring), d_taps, d_block, d_out, d_hdr, ring_len,
                      ld_block, n, ld_out, pos, out_lo, n_taps, w_lo, w_hi, 0, block_type,
                      out_type, close ? 1 : 0, hdr_words};
  return launch_stream<float>(a, n_chans, n_grid, s);
}

int parrm_stream_push(void* d_ring, int64_t n_chans, int64_t max_chunk, const int32_t* d_taps,
                      int32_t n_taps, int32_t w_min, int32_t w_max, const void* d_block,
                      int block_type, int64_t ld_block, int64_t n, void* d_out, int out_type,
                      int64_t ld_out, int64_t pos, const int64_t* d_pos, int close, int dtype,
                      void* stream) {
  PARRM_NVTX("parrm_stream_push");
  using namespace parrm;
  PARRM_REQUIRE(max_chunk >= 1, "parrm_stream_push: max_chunk must be >= 1");
  PARRM_REQUIRE(n >= 0 && n <= max_chunk,
                "parrm_stream_push: block of %lld samples is longer than the ring allows "
                "(max_chunk %lld)", (long long)n, (long long)max_chunk);
  PARRM_REQUIRE(pos >= 0, "parrm_stream_push: position %lld goes backwards past the stream start",
                (long long)pos);
  PARRM_REQUIRE(pos <= INT64_MAX / 2, "parrm_stream_push: position %lld out of range",
                (long long)pos);
  // one tap set for the whole stream: the ring of parrm_stream_ring_bytes and the first output
  // that follows from the position
  const int64_t lat = stream_latency(w_min);
  const int64_t out_lo = pos - lat > 0 ? pos - lat : 0;
  const int64_t n_grid = n + (close ? lat : 0);  // grid extent; independent of pos
  return stream_push_impl("parrm_stream_push", d_ring, stream_span(w_min, w_max) + max_chunk,
                          n_chans, d_taps, n_taps, w_min, w_max, d_block, block_type, ld_block,
                          n, d_out, out_type, ld_out, pos, out_lo, n_grid, d_pos, 1, close, dtype,
                          stream);
}

int parrm_stream_push_at(void* d_ring, int64_t ring_len, int64_t n_chans, const int32_t* d_taps,
                         int32_t n_taps, int32_t w_min, int32_t w_max, const void* d_block,
                         int block_type, int64_t ld_block, int64_t n, void* d_out, int out_type,
                         int64_t ld_out, int64_t pos, int64_t out_lo, const int64_t* d_hdr,
                         int close, int dtype, void* stream) {
  PARRM_NVTX("parrm_stream_push_at");
  using namespace parrm;
  const char* fn = "parrm_stream_push_at";
  PARRM_REQUIRE(n >= 0, "%s: negative block length %lld", fn, (long long)n);
  PARRM_REQUIRE(pos >= 0 && pos <= INT64_MAX / 2, "%s: position %lld out of range", fn,
                (long long)pos);
  PARRM_REQUIRE(out_lo >= 0 && out_lo <= pos,
                "%s: first output %lld outside [0, pos = %lld]", fn, (long long)out_lo,
                (long long)pos);
  PARRM_REQUIRE(n_taps >= 1 && w_min <= w_max, "%s: empty or unordered tap list", fn);
  PARRM_REQUIRE(ring_len >= 1, "%s: ring length %lld must be >= 1", fn, (long long)ring_len);
  // every sample this launch reads, [max(0, out_lo - w_max), pos + n), spans at most the ring:
  // all of it is still there and no slot written here is read here
  const int64_t oldest = out_lo - (w_max > 0 ? w_max : 0);
  const int64_t reach = pos + n - (oldest > 0 ? oldest : 0);
  PARRM_REQUIRE(reach <= ring_len,
                "%s: the push reads %lld samples back from pos + n, more than the ring of %lld "
                "holds (a shorter block, or a longer ring)", fn, (long long)reach,
                (long long)ring_len);
  const int64_t out_hi = stream_out_hi(pos + n, out_lo, stream_latency(w_min), close);
  const int64_t n_grid = n > out_hi - out_lo ? n : out_hi - out_lo;
  return stream_push_impl(fn, d_ring, ring_len, n_chans, d_taps, n_taps, w_min, w_max, d_block,
                          block_type, ld_block, n, d_out, out_type, ld_out, pos, out_lo, n_grid,
                          d_hdr, 2, close, dtype, stream);
}

int parrm_stream_window(const void* d_ring, int64_t ring_len, int64_t n_chans, int64_t pos,
                        int64_t n, void* d_dst, int64_t ld_dst, int dtype, void* stream) {
  PARRM_NVTX("parrm_stream_window");
  using namespace parrm;
  const char* fn = "parrm_stream_window";
  PARRM_REQUIRE(dtype == PARRM_F64 || dtype == PARRM_F32, "%s: bad dtype %d", fn, dtype);
  PARRM_REQUIRE(n_chans >= 1, "%s: need channels >= 1, got %lld", fn, (long long)n_chans);
  PARRM_REQUIRE(ring_len >= 1, "%s: ring length %lld must be >= 1", fn, (long long)ring_len);
  PARRM_REQUIRE(n >= 1 && n <= pos && n <= ring_len,
                "%s: window of %lld samples outside [1, min(pos = %lld, ring = %lld)]", fn,
                (long long)n, (long long)pos, (long long)ring_len);
  PARRM_REQUIRE(d_ring != nullptr && d_dst != nullptr && ld_dst >= n,
                "%s: null ring or destination, or row stride %lld < %lld", fn, (long long)ld_dst,
                (long long)n);
  // samples [pos - n, pos) sit in slots [first, first + n) mod R: two column ranges at most
  const size_t es = dtype == PARRM_F64 ? 8 : 4;
  const int64_t first = (pos - n) % ring_len;
  const int64_t n1 = n < ring_len - first ? n : ring_len - first;
  cudaStream_t s = as_stream(stream);
  const char* ring = static_cast<const char*>(d_ring);
  char* dst = static_cast<char*>(d_dst);
  PARRM_CUDA_OK(cudaMemcpy2DAsync(dst, size_t(ld_dst) * es, ring + size_t(first) * es,
                                  size_t(ring_len) * es, size_t(n1) * es, size_t(n_chans),
                                  cudaMemcpyDeviceToDevice, s));
  if (n1 < n)
    PARRM_CUDA_OK(cudaMemcpy2DAsync(dst + size_t(n1) * es, size_t(ld_dst) * es, ring,
                                    size_t(ring_len) * es, size_t(n - n1) * es, size_t(n_chans),
                                    cudaMemcpyDeviceToDevice, s));
  return PARRM_OK;
}

}  // extern "C"
