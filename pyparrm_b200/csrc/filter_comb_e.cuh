// Comb filter, "pattern first" form: body of PARRM.filter_data (parrm.py:861-869) for tap
// sets with comb structure (filter_plan.h), specialised at run time for one plan.
//
// This file is compiled twice: by nvcc with the defaults below (the cfg2 plan; build check,
// SASS inspection) and by NVRTC from filter_jit.cu with every PE_* macro set from the plan, so
// that the stride, the box lengths and every tap offset are immediates.
//
// The plan writes the tap sum as comb boxes over one stride d,
//     sum_{w in taps} x[t-w] = sum_k sum_b sum_{q<M_k} x[t - a_kb - q d]  +/- single taps + c x[t].
// Summing over the boxes first gives a short pattern  E_k[i] = sum_b x[i - a_kb]  (NB_k loads)
// and the comb becomes a running sum of E_k along the chain t, t+d, t+2d, ...:
//     S_k[t] = sum_{q<M_k} E_k[t - q d],     S_k[t + d] = S_k[t] + E_k[t + d] - E_k[t + d - M_k d].
// One thread owns one chain (one residue of t mod d).  It keeps the last M_k values of E_k in
// REGISTERS (statically indexed: the step loop is unrolled >= M_0 deep), so per output the shared
// memory pipe sees only the NB_0 + NB_1 pattern loads, the single taps and x[t] -- for the
// cfg2 filter (160 taps) 12 loads instead of 160, and no intermediate array at all.  The sums
// are re-added from the register rings once per unrolled block, which bounds rounding drift.
//
// Data movement: a persistent CTA walks a strip of consecutive chunks (U*d samples) of one
// channel.  A producer warp streams chunks HBM -> shared ring with TMA bulk copies
// (cp.async.bulk + mbarrier complete_tx; every sample is read from HBM once per strip); the
// first MIR ring chunks are mirrored behind the ring so the window a step reads is contiguous
// and every load is  [chain pointer + immediate].  D/32 consumer warps wait on the `full`
// barrier of the newest chunk, run U steps, and release the oldest chunk (`empty`).  Outputs
// go straight from registers to HBM, 32 consecutive samples per warp store.
//
// Non-finite samples: an output whose tap window (or own sample) holds a NaN/Inf is 0, as the
// reference's isfinite -> 0 replacement (parrm.py:869) intends (run_block: the sums are re-added
// from the rings while the bad value is inside the window, so outputs past it are exact again).
#pragma once

#ifdef __CUDACC_RTC__
typedef signed char int8_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
typedef unsigned long long uintptr_t;
#else
#include <stdint.h>
#endif

#ifndef PE_D  // defaults: BASELINE cfg2 (period 2000/130 samples, half width 2000, both directions)
#define PE_T double
#define PE_D 200
#define PE_NK 2
#define PE_M0 20
#define PE_M1 10
#define PE_NB0 7
#define PE_NB1 2
#define PE_OFF0 -1969, -1954, -1923, -1877, -1846, -1831, -1800
#define PE_OFF1 -1908, 108
#define PE_NPLUS 1
#define PE_PLUS -2000
#define PE_NMINUS 0
#define PE_MINUS 0
#define PE_CENTRE -1
#define PE_U 10
#define PE_PF 2
#define PE_NTAPS 160
#define PE_WLO -2000
#define PE_WHI 2000
#define PE_BACK 108
#define PE_FWD 2000
#define PE_CTAS 2
#endif
#ifndef PE_VARIANT
#define PE_VARIANT 0  // filter options: 2 = per-CTA timeline (profiling aid); 4 = strips of
                      // equal length instead of equal cost (host side, A/B)
#endif

namespace parrm_e {

typedef PE_T T;
typedef double T2;
constexpr int D = PE_D;            // comb stride = chains per strip
constexpr int NK = PE_NK;          // box lengths in use (1 or 2), M0 >= M1
constexpr int M0 = PE_M0;
constexpr int M1 = PE_M1;
constexpr int NB0 = PE_NB0;
constexpr int NB1 = PE_NB1;
constexpr int NPLUS = PE_NPLUS;
constexpr int NMINUS = PE_NMINUS;
constexpr int CENTRE = PE_CENTRE;  // coefficient of x[t] inside the tap sum (<= 0)
constexpr int U = PE_U;            // steps per chunk
constexpr int PF = PE_PF;          // chunks in flight beyond the window
constexpr int NTAPS = PE_NTAPS;
constexpr int WLO = PE_WLO;        // min(w_min, 0)
constexpr int WHI = PE_WHI;        // max(w_max, 0)
constexpr int BACK = PE_BACK;      // largest offset any load reaches back from t (>= 0)
constexpr int FWD = PE_FWD;        // ... forward (>= 0)
constexpr int ES = int(sizeof(T));
constexpr int VEC = 16 / ES;
constexpr int CH = U * D;                        // samples per chunk
constexpr int HB = (BACK + CH - 1) / CH;         // chunks behind the current one a step reads
constexpr int HF = (FWD + CH - 1) / CH;          // chunks ahead
constexpr int MIR = HB + HF;                     // mirrored ring chunks
constexpr int Q = HB + HF + 1 + PF;              // ring chunks
constexpr int GPB = (M0 + U - 1) / U;            // groups (chunks) per unrolled block
constexpr int B = GPB * U;                       // steps per unrolled block (>= M0)
constexpr int NPG = GPB;                         // priming groups: one block fills the rings
constexpr int NW = (D + 31) / 32;                // consumer warps
constexpr int NT = NW * 32 + 32;                 // + one producer warp
constexpr int BAR_BYTES = ((2 * Q * 8 + 127) / 128) * 128;
constexpr int SMEM_BYTES = BAR_BYTES + (Q + MIR) * CH * ES;
static_assert((CH * ES) % 16 == 0, "chunk must be a whole number of 16-byte units");
static_assert(M0 >= M1 && M0 >= 1, "box lengths ordered");

// tap offsets of the plan (compile-time tables; every use folds to an immediate)
__host__ __device__ constexpr int off0(int b) {
  constexpr int t[NB0 > 0 ? NB0 : 1] = {PE_OFF0};
  return t[b];
}
__host__ __device__ constexpr int off1(int b) {
  constexpr int t[NB1 > 0 ? NB1 : 1] = {PE_OFF1};
  return t[b];
}
__host__ __device__ constexpr int plus_tap(int i) {
  constexpr int t[NPLUS > 0 ? NPLUS : 1] = {PE_PLUS};
  return t[i];
}
__host__ __device__ constexpr int minus_tap(int i) {
  constexpr int t[NMINUS > 0 ? NMINUS : 1] = {PE_MINUS};
  return t[i];
}

struct Args {
  const T* x;
  T* out;
  const int32_t* taps;   // plan: the NTAPS tap offsets, ascending (rare path only)
  const int32_t* count;  // plan table: count[v - (WLO - 1)] = #{taps <= v}, WLO - 1 <= v <= WHI
  const T2* recip;       // plan table: 0, 1/1, 1/2, ... 1/NTAPS (float64)
  int64_t ld_x, x_t0, n_x;
  int64_t ld_out, t0, n_out;
  int64_t n_total;
  int64_t total_groups;  // n_chans * (groups_per_chan + edge_total): the cost units CTAs share
  int32_t groups_per_chan;
  int32_t edge_start;    // cost of starting a channel (priming, window fill, edge blocks), in groups
  int32_t edge_total;    // ... of starting and ending it
  int32_t pad;
  unsigned long long* timeline;  // profiling aid (PE_VARIANT & 2): 4 words per CTA, or null
  T neg_inv_n;  // -1 / NTAPS   (kernel parameters: FP64 instructions take them as constant-bank
  T t_max;      // largest finite T           operands, so they occupy no registers in the loop)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ int64_t floor_div(int64_t a, int64_t b) {
  int64_t q = a / b;
  return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q;
}
__device__ __forceinline__ int64_t min64(int64_t a, int64_t b) { return a < b ? a : b; }
__device__ __forceinline__ int64_t max64(int64_t a, int64_t b) { return a > b ? a : b; }

// Recording edges (outputs whose tap window leaves [0, n_total), and chunks only partly inside
// the requested output range): mean over the in-range taps, parrm.py:861-866.  The number of
// in-range taps  #{w : 0 <= t - w < n_total} = #{w <= t} - #{w <= t - n_total}  comes from the
// plan's cumulative table, its reciprocal from the plan's reciprocal table (no search, no
// division: this sits in the unrolled step loop and must stay small).
__device__ __forceinline__ T edge_value(const int32_t* __restrict__ count,
                                        const T2* __restrict__ recip, int64_t t, int64_t n_total,
                                        T xc, T tot) {
  const int64_t v1 = min64(max64(t, WLO - 1), WHI);
  const int64_t v2 = min64(max64(t - n_total, WLO - 1), WHI);
  const int n_in = count[v1 - (WLO - 1)] - count[v2 - (WLO - 1)];
  T y = xc - tot * T(recip[n_in]);
  if (n_in == 0) y = T(0);
  return y;
}

// Rare path: an output whose fast value came out non-finite is re-evaluated tap by tap from
// global memory, exactly as the definition reads (parrm.py:861-869): mean over the in-range
// taps, 0 when that is not finite.  This is what makes a NaN / Inf sample zero exactly the
// outputs whose tap window (or own sample) holds it, even where the plan covers a non-tap
// offset with a box and cancels it with a -1 term (NaN - NaN does not cancel).  It runs after
// the piece, over the span of steps the step loop flagged, so that the loop itself holds no
// call (a call in a cold branch still makes the compiler rebuild addresses after the join).
// (Everything by value: taking the address of the kernel's parameter struct would move it from
// the constant bank to local memory for the whole kernel.)
__device__ __noinline__ T direct_value(const int32_t* __restrict__ taps,
                                       const T2* __restrict__ recip, int64_t n_total, T t_max,
                                       const T* __restrict__ xrow, int64_t t, int64_t lo_valid,
                                       int64_t hi_valid) {
  T acc = T(0);
  int n_in = 0;
  for (int k = 0; k < NTAPS; ++k) {
    const int64_t g = t - taps[k];
    if (g < 0 || g >= n_total) continue;
    ++n_in;
    if (g >= lo_valid && g < hi_valid) acc += xrow[g];
  }
  if (n_in == 0) return T(0);
  const T y = xrow[t] - acc * T(recip[n_in]);
  return fabs(y) <= t_max ? y : T(0);
}

// A consumer thread's position in the chunk sequence of its piece.
struct Walk {
  int pb;           // byte offset (from smem_raw) of the sample HB*CH before the group's first output
  int rslot;        // oldest live ring slot (next to release)
  int fslot;        // next ring slot to wait for
  uint32_t fphase;  // parity of that fill
};

// Opens a group: its newest chunk has landed.
__device__ __forceinline__ void group_begin(Walk& w, uint32_t bars) {
  mbar_wait(bars + w.fslot * 8, w.fphase);
  if (++w.fslot == Q) {
    w.fslot = 0;
    w.fphase ^= 1u;
  }
}
// Closes a group: its oldest chunk is released to the producer.
__device__ __forceinline__ void group_end(Walk& w, uint32_t bars, int lane, unsigned wmask) {
  __syncwarp(wmask);
  if (lane == 0) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bars + (Q + w.rslot) * 8)
                 : "memory");
  }
  w.pb += CH * ES;
  if (++w.rslot == Q) {
    w.rslot = 0;
    w.pb -= Q * CH * ES;
  }
}

// Register rings of one chain: the last M_k pattern values, statically indexed.  The step
// loop is unrolled B = U * ceil(M0 / U) deep (a whole number of chunks, so chunk boundaries
// sit at fixed places of the unrolled code); ring position s of a block is written at step s
// and read again M_k steps later, so only M_0 + M_1 entries are live at any time.
struct Rings {
  T r0[B];
  T r1[NK > 1 ? B : 1];
  T S0, S1;
};

// sum of the last M_k ring entries, the newest at position s (static after unrolling)
__device__ __forceinline__ T ring_sum0(const Rings& r, int s) {
  T a = r.r0[s];
#pragma unroll
  for (int i = 1; i < M0; ++i) a += r.r0[(s + B - i) % B];
  return a;
}
__device__ __forceinline__ T ring_sum1(const Rings& r, int s) {
  if (NK < 2) return T(0);
  T a = r.r1[s];
#pragma unroll
  for (int i = 1; i < M1; ++i) a += r.r1[(s + B - i) % B];
  return a;
}

// One block of B steps (GPB groups) of one chain.  FAST: every output of the block is an
// interior output inside the requested range -- no per-group mode, no edge code.  Otherwise
// groups may be priming groups (no outputs), recording edges or partial ranges, and the piece
// may end inside the block.  Returns the number of groups done.
//
// Non-finite samples: the fast path only tests the finished output.  A NaN/Inf that entered a
// running sum keeps it non-finite, so the test fails on every step until the bad pattern
// value has left the ring; on those (rare) steps the sums are re-added from the rings (which
// makes the first output past the window exact again) and the output itself is re-evaluated
// tap by tap (direct_value).
template <bool FAST>
__device__ __forceinline__ int run_block(Rings& r, Walk& w, const Args& a,
                                         const unsigned char* const smem, uint32_t bars,
                                         int lane, unsigned wmask, int c, T* const orow,
                                         int& bad_lo, int& bad_hi, int64_t Tb, int g,
                                         int n_groups) {
  const T neg_inv_n = a.neg_inv_n;
  const T t_max = a.t_max;
  T* const op = orow + Tb + c;  // output of step 0 of the block
  int done = 0;
#pragma unroll
  for (int gi = 0; gi < GPB; ++gi) {
    if (!FAST && g + gi >= n_groups) break;
    group_begin(w, bars);
    int mode = 1;  // 0 priming (no outputs), 1 interior, 2 recording edge / partial range
    if (!FAST) {
      const int64_t Tn = Tb + int64_t(gi) * CH;
      const bool interior = (Tn - WHI >= 0) && (Tn + CH - WLO <= a.n_total);
      const bool all_out = (Tn >= a.t0) && (Tn + CH <= a.t0 + a.n_out);
      mode = (g + gi < NPG) ? 0 : ((interior && all_out) ? 1 : 2);
    }
    const unsigned char* const p = smem + w.pb;
#pragma unroll
    for (int js = 0; js < U; ++js) {
      const int s = gi * U + js;
      auto ld = [&](int off) {  // sample at (current output time - off)
        return *reinterpret_cast<const T*>(p + (HB * CH + js * D - off) * ES);
      };
      // leaving values first: their registers are free for the new pattern values
      r.S0 -= r.r0[(s + B - M0) % B];
      if (NK > 1) r.S1 -= r.r1[(s + B - M1) % B];
      T e0 = ld(off0(0));  // two partial sums: shorter dependent chains
      if (NB0 > 1) {
        T e0b = ld(off0(1));
#pragma unroll
        for (int b = 2; b < NB0; ++b) {
          if (b & 1) e0b += ld(off0(b)); else e0 += ld(off0(b));
        }
        e0 += e0b;
      }
      r.r0[s] = e0;
      r.S0 += e0;
      T tot = r.S0;
      if (NK > 1) {
        T e1 = ld(off1(0));
        if (NB1 > 1) {
          T e1b = ld(off1(1));
#pragma unroll
          for (int b = 2; b < NB1; ++b) {
            if (b & 1) e1b += ld(off1(b)); else e1 += ld(off1(b));
          }
          e1 += e1b;
        }
        r.r1[s] = e1;
        r.S1 += e1;
        tot += r.S1;
      }
      T single = T(0);
      if (NPLUS > 0) {
        single = ld(plus_tap(0));
#pragma unroll
        for (int i = 1; i < NPLUS; ++i) single += ld(plus_tap(i));
      }
#pragma unroll
      for (int i = 0; i < NMINUS; ++i) single -= ld(minus_tap(i));
      const T xc = ld(0);
      if (CENTRE != 0) single = fma(T(CENTRE), xc, single);
      if (NPLUS > 0 || NMINUS > 0 || CENTRE != 0) tot += single;
      if (FAST) {
        T y = fma(tot, neg_inv_n, xc);
        if (__builtin_expect(!(fabs(y) <= t_max), 0)) {
          r.S0 = ring_sum0(r, s);
          r.S1 = ring_sum1(r, s);
          bad_lo = min(bad_lo, g * U + s);
          bad_hi = max(bad_hi, g * U + s);
          y = T(0);
        }
        op[s * D] = y;
      } else if (mode != 0) {
        const int64_t t = Tb + c + int64_t(s) * D;
        if (ES == 4 && mode == 2) {
          // float32 at a recording edge: the sums are re-added from the rings on every step.
          // Where the window runs off the end of the recording, n_in falls to 1 while a running
          // sum still carries the rounding of up to 2B updates of the full window (~n_taps |x|
          // each) since the block began; divided by n_in that is ~2B n_taps eps32 |x|, above
          // 1e-4 of the input scale for the cfg4 taps.  Re-added, only the rounding of the
          // in-range values is left.  (float64 keeps the running sums: 2^-29 times smaller.)
          r.S0 = ring_sum0(r, s);
          r.S1 = ring_sum1(r, s);
          tot = r.S0;
          if (NK > 1) tot += r.S1;
          if (NPLUS > 0 || NMINUS > 0 || CENTRE != 0) tot += single;
        }
        T y = mode == 1 ? fma(tot, neg_inv_n, xc) : edge_value(a.count, a.recip, t, a.n_total, xc, tot);
        if (__builtin_expect(!(fabs(y) <= t_max), 0)) {
          r.S0 = ring_sum0(r, s);
          r.S1 = ring_sum1(r, s);
          bad_lo = min(bad_lo, g * U + s);
          bad_hi = max(bad_hi, g * U + s);
          y = T(0);
        }
        if (t >= a.t0 && t < a.t0 + a.n_out) op[s * D] = y;
      }
    }
    group_end(w, bars, lane, wmask);
    ++done;
  }
  return done;
}

extern "C" __global__ void __launch_bounds__(NT, PE_CTAS) parrm_filter_comb_e(const Args a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* const full = reinterpret_cast<uint64_t*>(smem_raw);  // [Q] chunk landed
  uint64_t* const empty = full + Q;                              // [Q] chunk released
  T* const ring = reinterpret_cast<T*>(smem_raw + BAR_BYTES);    // (Q + MIR) chunks
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const bool is_producer = tid >= NW * 32;

  if (tid == 0) {
    for (int s = 0; s < Q; ++s) {
      mbar_init(&full[s], 1);    // the producer's elected lane arrives (plus the TMA bytes)
      mbar_init(&empty[s], NW);  // one lane of every consumer warp arrives
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const int64_t lo_valid = max64(0, a.x_t0);
  const int64_t hi_valid = min64(a.n_total, a.x_t0 + a.n_x);
#if PE_VARIANT & 2
  unsigned long long tl_start = 0, tl_pieces = 0;
  if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tl_start));
#endif
  const int gpc = a.groups_per_chan;
  // Strips of equal COST, not equal length: a strip that crosses a channel boundary pays a
  // second priming block, a second window fill and the slower generic blocks of both recording
  // edges (measured per CTA, scripts/filter_timeline.py: +18 us on 238 us at the cfg2 shape,
  // and the kernel ends with its slowest CTA).  Every channel is therefore edge_total cost
  // units longer than its groups, edge_start of them in front.
  const int vpc = gpc + a.edge_total;
  const int64_t G_begin = a.total_groups * int64_t(blockIdx.x) / int64_t(gridDim.x);
  const int64_t G_end = a.total_groups * int64_t(blockIdx.x + 1) / int64_t(gridDim.x);
  const uint32_t bars = smem_u32(smem_raw);

  // Chunks are numbered by one counter that runs on through all pieces of this CTA: chunk
  // number s lives in ring slot s % Q and is the (s / Q)-th fill of that slot.  Both roles
  // keep (slot, phase) of their own position in that sequence.
  int fslot = 0;        // producer: next slot to fill;  consumer: next slot to wait for
  uint32_t fphase = 0;  // parity of that fill
  int rslot = 0;        // consumer: oldest live slot (next to release)

  for (int64_t G = G_begin; G < G_end;) {
    const int64_t chan = G / vpc;
    const int v0 = int(G - chan * vpc);
    const int v1 = int(min64(vpc, v0 + (G_end - G)));
    G += v1 - v0;
    const int s0 = min(max(v0 - a.edge_start, 0), gpc);
    const int s1 = min(max(v1 - a.edge_start, 0), gpc);
    if (s1 <= s0) continue;
    const T* const xrow = a.x + chan * a.ld_x - a.x_t0;  // xrow[g] = sample at global time g
    T* const orow = a.out + chan * a.ld_out - a.t0;      // orow[g]
    const int gamma = int((VEC - int((reinterpret_cast<uintptr_t>(xrow) / ES) % VEC)) % VEC);
    const int64_t j_first = floor_div(a.t0 - gamma, CH);
    const int64_t j_last = floor_div(a.t0 + a.n_out - 1 - gamma, CH);
    const int64_t n_first = j_first + s0;                      // first group with outputs
    const int64_t n_end = min64(j_first + s1, j_last + 1);
    if (n_first >= n_end) continue;
#if PE_VARIANT & 2
    ++tl_pieces;
#endif
    const int n_groups = NPG + int(n_end - n_first);           // priming groups first
    const int n_chunks = n_groups + HB + HF;
    const int64_t c_first = n_first - NPG - HB;                // first chunk the piece reads

    if (is_producer) {
      // ------------------------------ producer warp ------------------------------
      for (int i = 0; i < n_chunks; ++i) {
        const int64_t g0 = gamma + (c_first + i) * int64_t(CH);
        T* const dst = ring + fslot * CH;
        // (a nanosleep back-off in this wait was measured: no gain with two CTAs per SM, and
        // -15 % with one, where a late refill stalls every consumer warp)
        mbar_wait(bars + (Q + fslot) * 8, fphase ^ 1u);  // the previous fill has been released
        if (g0 >= lo_valid && g0 + CH <= hi_valid) {
          if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            const bool mirror = fslot < MIR;
            mbar_expect_tx(&full[fslot], uint32_t(CH * ES) * (mirror ? 2u : 1u));
            bulk_g2s(dst, xrow + g0, uint32_t(CH * ES), &full[fslot]);
            if (mirror) bulk_g2s(dst + Q * CH, xrow + g0, uint32_t(CH * ES), &full[fslot]);
          }
        } else {  // chunk crosses an end of the available samples: zero fill
          for (int e = lane; e < CH; e += 32) {
            const int64_t g = g0 + e;
            const T v = (g >= lo_valid && g < hi_valid) ? xrow[g] : T(0);
            dst[e] = v;
            if (fslot < MIR) dst[Q * CH + e] = v;
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&full[fslot]);
        }
        if (++fslot == Q) {
          fslot = 0;
          fphase ^= 1u;
        }
      }
      continue;
    }

    // ------------------------------ consumer warps ------------------------------
    // Lanes past the last chain idle: a half-warp with no active lane costs the shared-memory
    // pipe no wavefront (D = 200: 1 of 14 wavefronts per load instruction of the CTA).
    if (tid >= D) continue;
    const int c = tid;
    const unsigned wmask = (tid | 31) < D ? 0xffffffffu : ((1u << (D & 31)) - 1u);
    for (int i = 0; i < HB + HF; ++i) {   // the window of the first group, except its newest chunk
      mbar_wait(bars + fslot * 8, fphase);
      if (++fslot == Q) {
        fslot = 0;
        fphase ^= 1u;
      }
    }
    Rings r;
#pragma unroll
    for (int s = 0; s < B; ++s) r.r0[s] = T(0);
#pragma unroll
    for (int s = 0; s < (NK > 1 ? B : 1); ++s) r.r1[s] = T(0);
    const int64_t T0 = gamma + (n_first - NPG) * int64_t(CH);  // time of the piece's first group
    Walk w;
    w.pb = BAR_BYTES + (rslot * CH + c) * ES;
    w.rslot = rslot;
    w.fslot = fslot;
    w.fphase = fphase;
    int bad_lo = 1 << 30, bad_hi = -1;  // span of steps whose fast output was not finite
    for (int g = 0; g < n_groups;) {
      const int64_t Tb = T0 + int64_t(g) * CH;
      // fresh sums from the rings (bounds the drift of the running update)
      r.S0 = ring_sum0(r, B - 1);
      r.S1 = ring_sum1(r, B - 1);
      const bool fast = g >= NPG && g + GPB <= n_groups && Tb - WHI >= 0 &&
                        Tb + int64_t(B) * D - WLO <= a.n_total && Tb >= a.t0 &&
                        Tb + int64_t(B) * D <= a.t0 + a.n_out;
      if (fast) {
        g += run_block<true>(r, w, a, smem_raw, bars, lane, wmask, c, orow, bad_lo, bad_hi,
                             Tb, g, n_groups);
      } else {
        g += run_block<false>(r, w, a, smem_raw, bars, lane, wmask, c, orow, bad_lo, bad_hi,
                              Tb, g, n_groups);
      }
    }
    rslot = w.rslot;
    fslot = w.fslot;
    fphase = w.fphase;
    for (int k = bad_lo; k <= bad_hi; ++k) {  // rare: re-evaluate the flagged span by the definition
      const int64_t t = T0 + c + int64_t(k) * D;
      if (t >= a.t0 && t < a.t0 + a.n_out)
        orow[t] = direct_value(a.taps, a.recip, a.n_total, a.t_max, xrow, t, lo_valid, hi_valid);
    }
    // release the rest of the window (chunks the last group still held)
    __syncwarp(wmask);
    for (int i = 0; i < HB + HF; ++i) {
      if (lane == 0) mbar_arrive(&empty[rslot]);
      if (++rslot == Q) rslot = 0;
    }
  }
#if PE_VARIANT & 2
  if (tid == 0 && a.timeline) {
    unsigned long long tl_end;
    unsigned smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tl_end));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    a.timeline[4 * blockIdx.x + 0] = smid;
    a.timeline[4 * blockIdx.x + 1] = tl_start;
    a.timeline[4 * blockIdx.x + 2] = tl_end;
    a.timeline[4 * blockIdx.x + 3] = tl_pieces;
  }
#endif
}

}  // namespace parrm_e
