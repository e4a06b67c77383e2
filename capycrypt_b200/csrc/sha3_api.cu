// sha3_api.cu -- SHA3-d / cSHAKE / KMACXOF batch entry points (C ABI in include/capy_gpu.h).
//
// Replaces, for batches, the reference call stack
//   hashable.rs:19-35 -> shake_functions.rs:24-89 -> sponge.rs:10-34 -> keccakf.rs:8-423.
// The SP 800-185 encoders (aux_functions.rs:11-68) run on the host only to build the constant
// prefix block of cSHAKE/KMAC; every byte that is absorbed per item is produced on the device.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <memory>
#include <thread>
#include <type_traits>
#include <vector>

#include "internal.h"
#include "hostbatch.h"
#include "keccak_bs.cuh"
#include "sponge.cuh"

namespace capy {

// ------------------------------------------------------------------------------------------------
// uniform-length SHA3-d kernel: every message has the same length, 8-byte aligned starts.
// All control flow depends only on (len, LANES) so it is warp-uniform; the message bytes go
// straight from global memory into the state registers.  This is the cfg-1 hot kernel
// (2^20 x 64 B: one permutation, 4 x 16 B loads, 2 x 16 B stores per thread).
// ------------------------------------------------------------------------------------------------
template <int LANES>
__global__ void __launch_bounds__(128)
    sha3_uniform_kernel(const uint8_t* __restrict__ data, uint64_t stride, uint64_t len, uint32_t suffix,
                        uint8_t* __restrict__ out, uint32_t out_bytes, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  constexpr uint64_t RATE = 8ull * LANES;
  const uint2* q = reinterpret_cast<const uint2*>(data + i * stride);
  Lane a[25];
  state_zero(a);
  const uint64_t nfull = len / RATE;
  for (uint64_t b = 0; b < nfull; b++) {
#pragma unroll
    for (int j = 0; j < LANES; j++) {
      uint2 v = __ldg(q + j);
      a[j].lo ^= v.x;
      a[j].hi ^= v.y;
    }
    q += LANES;
    keccak_f1600(a);
  }
  // final block: rem message bytes, the suffix byte, then (only if rem + 1 < RATE) zeros..0x80
  const uint32_t rem = (uint32_t)(len - nfull * RATE);
#pragma unroll
  for (int j = 0; j < LANES; j++) {
    const uint32_t o = 8u * j;
    uint32_t lo = 0, hi = 0;
    if (o < rem) {  // the aligned 8-byte word holds at least one message byte
      uint2 v = __ldg(q + j);
      lo = v.x;
      hi = v.y;
      if (o + 8 > rem) {  // partial lane: keep rem - o bytes
        const uint32_t keep = rem - o;  // 1..7
        if (keep < 4) {
          lo &= (1u << (8 * keep)) - 1u;
          hi = 0;
        } else if (keep > 4) {
          hi &= (1u << (8 * (keep - 4))) - 1u;
        } else {
          hi = 0;
        }
      }
    }
    if (rem >= o && rem < o + 8) {
      const uint32_t k = rem - o;
      if (k < 4) lo |= suffix << (8 * k);
      else hi |= suffix << (8 * (k - 4));
    }
    a[j].lo ^= lo;
    a[j].hi ^= hi;
  }
  if (rem + 1 < RATE) a[LANES - 1].hi ^= 0x80000000u;  // quirk Q1: no 0x80 when already aligned
  keccak_f1600(a);

  uint8_t* o = out + i * (uint64_t)out_bytes;
  if ((out_bytes & 15u) == 0 && (reinterpret_cast<uintptr_t>(out) & 15u) == 0) {
#pragma unroll
    for (int j = 0; j < 4; j++)
      if (16u * j < out_bytes)
        reinterpret_cast<uint4*>(o)[j] = make_uint4(a[2 * j].lo, a[2 * j].hi, a[2 * j + 1].lo, a[2 * j + 1].hi);
  } else {  // 28- and 48-byte digests: 4-byte granules
#pragma unroll
    for (int j = 0; j < 8; j++) {
      if (8u * j < out_bytes) reinterpret_cast<uint32_t*>(o)[2 * j] = a[j].lo;
      if (8u * j + 4 < out_bytes) reinterpret_cast<uint32_t*>(o)[2 * j + 1] = a[j].hi;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// single-block SHA3-d of messages of exactly 8 * MSG_LANES bytes (MSG_LANES < LANES), 16-byte aligned
// rows: the BASELINE cfg-1 shape (2^20 x 64 B).  Bitsliced (keccak_bs.cuh): a warp hashes its 32 messages together,
// so the rotations run on the shuffle unit instead of the ALU pipe.  Each thread loads its own row with 128-bit loads;
// a warp transpose turns the message words into bit-position words.  Everything about the block layout is a
// compile-time constant: the zero lanes of the block fold away in the peeled round 0, the remaining 23 rounds run two
// per loop iteration, and round 23 computes only the digest lanes.
// Every thread of a warp that has a message takes part in every shuffle; threads past n hash zeros and store nothing.
// The minimum of 4 blocks per SM lets ptxas use up to 128 registers: under the plain bound it chose 96 and spilled.
// ------------------------------------------------------------------------------------------------
template <int LANES, int MSG_LANES>
__global__ void __launch_bounds__(128, 4)
    sha3_short_kernel(const uint4* __restrict__ data, uint64_t stride16, uint32_t suffix, uint4* __restrict__ out,
                      uint32_t out_bytes, uint64_t n) {
  static_assert(MSG_LANES % 2 == 0 && MSG_LANES < LANES, "whole 16-byte loads, one block");
  constexpr int OUT_LANES = (200 - 8 * LANES) / 16;  // d / 64: 4 (SHA3-256) or 8 (SHA3-512)
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i - lane >= n) return;  // warp-uniform: the warp has no message
  const bool live = i < n;
  const BsTranspose transpose(lane);

  uint32_t a[25][2];
  {
    const uint4* q = data + i * stride16;
    uint32_t w[2 * MSG_LANES];
#pragma unroll
    for (int j = 0; j < MSG_LANES / 2; j++) {
      const uint4 v = live ? __ldg(q + j) : make_uint4(0u, 0u, 0u, 0u);
      w[4 * j] = v.x;
      w[4 * j + 1] = v.y;
      w[4 * j + 2] = v.z;
      w[4 * j + 3] = v.w;
    }
#pragma unroll
    for (int j = 0; j < 2 * MSG_LANES; j++) w[j] = transpose(w[j]);
#pragma unroll
    for (int l = 0; l < MSG_LANES; l++) bs_gather(a[l], w[2 * l], w[2 * l + 1], lane);
  }
#pragma unroll
  for (int l = MSG_LANES; l < 25; l++) a[l][0] = a[l][1] = 0u;
  // 0x06 (0x86 can only occur for 135-byte messages, which are not 8-byte multiples): bits 2t, 2t+1 of the suffix
  const uint32_t pad = (uint32_t)((uint64_t)suffix >> (2 * lane));
  a[MSG_LANES][0] = 0u - (pad & 1u);
  a[MSG_LANES][1] = 0u - ((pad >> 1) & 1u);
  // 8 * MSG_LANES + 1 < rate always holds here: zeros then 0x80 (sponge.rs:89-95), bit 63 of the last lane
  a[LANES - 1][1] ^= lane == 31 ? 0xFFFFFFFFu : 0u;

  const uint2 rc = __ldg(&KECCAK_RC_BITS[lane]);
  keccak_bs_round(a, lane, rc, 1u);
#pragma unroll 1
  for (int r = 1; r < 23; r += 2) {
    keccak_bs_round(a, lane, rc, 1u << r);
    keccak_bs_round(a, lane, rc, 2u << r);
  }
  keccak_bs_round(a, lane, rc, 1u << 23);

  uint32_t w[2 * OUT_LANES];
#pragma unroll
  for (int l = 0; l < OUT_LANES; l++) bs_scatter(w[2 * l], w[2 * l + 1], a[l], lane);
#pragma unroll
  for (int j = 0; j < 2 * OUT_LANES; j++) w[j] = transpose(w[j]);
  if (!live) return;
  uint4* o = out + i * (uint64_t)(out_bytes / 16);
#pragma unroll
  for (int j = 0; j < OUT_LANES / 2; j++) o[j] = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
}

// one thread absorbs the whole-block part of a constant prefix into a cached state
template <int LANES>
__global__ void prefix_state_kernel(const uint8_t* prefix, uint32_t nblocks, uint64_t* state) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  Lane a[25];
  state_zero(a);
  for (uint32_t b = 0; b < nblocks; b++) {
    const uint8_t* p = prefix + (size_t)b * 8 * LANES;
#pragma unroll
    for (int j = 0; j < LANES; j++) {
      uint64_t v = 0;
      for (int k = 0; k < 8; k++) v |= (uint64_t)p[8 * j + k] << (8 * k);
      a[j].lo ^= (uint32_t)v;
      a[j].hi ^= (uint32_t)(v >> 32);
    }
    keccak_f1600(a);
  }
  for (int k = 0; k < 25; k++) state[k] = ((uint64_t)a[k].hi << 32) | a[k].lo;
}

// ------------------------------------------------------------------------------------------------
// Mixed-length batches (BASELINE config 5): longest-processing-time-first order.
// A sponge is sequential per message, so with one thread per message the job cannot finish before
// the longest message does.  Items are bucketed by block count (counting sort on the device) and
// processed longest first; when the longest chain would dominate, the launch is limited to 1-3 warps
// per scheduler (dynamic shared memory as an occupancy throttle) so that chain advances at full speed.
// ------------------------------------------------------------------------------------------------
// 16 384 bins of one block each; longer messages (>= 1.1 MB at the SHA3-512 rate) share the last bin
constexpr uint32_t kLenBins = 1u << 14;
constexpr uint64_t kHostPlanMaxItems = 1ull << 18;  // plan_ragged: largest batch whose histogram is taken on the host

__device__ __forceinline__ uint32_t len_bin(const uint64_t* off, uint64_t i, uint32_t stride_bytes) {
  const uint64_t blocks = (off[i + 1] - off[i]) / stride_bytes;
  return blocks < kLenBins - 1 ? (uint32_t)blocks : kLenBins - 1;
}

__global__ void len_hist_kernel(const uint64_t* __restrict__ off, uint64_t n, uint32_t stride_bytes, uint32_t* hist) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&hist[len_bin(off, i, stride_bytes)], 1u);
}

// hist[k] := number of items in bins > k (start of bin k in descending order); summary = {total blocks
// (lo, hi), max bin, number of non-empty bins}.  1024 threads x 16 consecutive bins (four 128-bit loads each),
// thread 0 owns the HIGHEST bins.
__global__ void __launch_bounds__(1024) len_scan_kernel(uint32_t* hist, uint32_t* summary) {
  __shared__ unsigned long long tot_s;
  __shared__ uint32_t max_s, bins_s;
  const uint32_t t = threadIdx.x;
  constexpr uint32_t PER = kLenBins / 1024;  // 16
  static_assert(PER == 16, "four uint4 per thread");
  if (t == 0) { tot_s = 0; max_s = 0; bins_s = 0; }
  __syncthreads();
  const uint32_t lo = kLenBins - (t + 1) * PER;  // this thread's bins lo .. lo + 15
  uint32_t c[PER];
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint4 v = reinterpret_cast<const uint4*>(hist + lo)[q];
    c[4 * q] = v.x; c[4 * q + 1] = v.y; c[4 * q + 2] = v.z; c[4 * q + 3] = v.w;
  }
  uint32_t sum = 0, nb = 0, mx = 0;
  unsigned long long tot = 0;
#pragma unroll
  for (int k = 0; k < (int)PER; k++) {
    sum += c[k];
    if (c[k]) { nb++; mx = lo + k; }  // ascending k: the last non-empty one is the largest
    tot += (unsigned long long)c[k] * (lo + k + 1);
  }
  if (sum) {
    atomicAdd(&tot_s, tot);
    atomicMax(&max_s, mx);
    atomicAdd(&bins_s, nb);
  }
  __syncthreads();
  // inclusive scan of the per-thread sums over the threads (thread 0 = highest bins): warp shuffles, then the 32 warp totals
  uint32_t incl = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
    if ((t & 31) >= (uint32_t)d) incl += v;
  }
  __shared__ uint32_t wsum[32];
  if ((t & 31) == 31) wsum[t >> 5] = incl;
  __syncthreads();
  if (t < 32) {
    uint32_t w = wsum[t];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, w, d);
      if (t >= (uint32_t)d) w += v;
    }
    wsum[t] = w;
  }
  __syncthreads();
  uint32_t run = incl - sum + ((t >> 5) ? wsum[(t >> 5) - 1] : 0u);  // items in bins above this thread's range
  // descending inside the thread: bin lo + 15 first
#pragma unroll
  for (int k = (int)PER - 1; k >= 0; k--) {
    const uint32_t cnt = c[k];
    c[k] = run;
    run += cnt;
  }
#pragma unroll
  for (int q = 0; q < 4; q++) reinterpret_cast<uint4*>(hist + lo)[q] = make_uint4(c[4 * q], c[4 * q + 1], c[4 * q + 2], c[4 * q + 3]);
  if (t == 0) {
    summary[0] = (uint32_t)tot_s;
    summary[1] = (uint32_t)(tot_s >> 32);
    summary[2] = max_s;
    summary[3] = bins_s;
  }
}

__global__ void len_scatter_kernel(const uint64_t* __restrict__ off, uint64_t n, uint32_t stride_bytes, uint32_t* cursor,
                                   uint32_t* __restrict__ order) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) order[atomicAdd(&cursor[len_bin(off, i, stride_bytes)], 1u)] = (uint32_t)i;
}

// Measured on B200, per permutation of ONE chain inside the sponge (tools/bench_tier_probe.py, 1 MiB SHA3-512 messages,
// profiles/README.md round 2): one thread per state 4.6 us; a thread pair 3.08 us; a whole warp per state 2.04 us on an
// otherwise idle GPU and 2.06 us with every SM busy.  A warp-tier chain issues only ~32 instructions per ~170-clock round,
// so several can share a scheduler -- but the 18 shuffles of its round go through one shuffle unit per SM (one warp-wide
// shuffle per clock): with c chains per scheduler a round cannot be shorter than 72 c clocks.  Measured: 2.06 / 2.36 /
// 3.0 us per permutation at c = 1 / 2 / 3.
constexpr double kPairChainRatio = 3.08 / 4.6;
constexpr int kMaxWarpCosched = 3;
constexpr double kWarpChainRatio[kMaxWarpCosched + 1] = {0.0, 2.06 / 4.6, 2.36 / 4.6, 3.00 / 4.6};

// Tiers of a chain-bound batch.  cum[k] = number of items in length bins > k (bin = whole blocks of the message).
// Times are in units of one thread-per-state permutation; an SM hosts ONE block: 4 c warp-tier items (c = 1, 2 or 3
// chains per scheduler), 64 pair-tier or 128 thread-tier items.  For a step time T every item takes the cheapest
// class its chain still fits: warp tier with a scheduler to itself for the longest, then two and three chains per
// scheduler, then the pair tier, the rest one thread per item.  The smallest T is taken for which (a) the blocks of the
// fast tiers are all resident from the start and (b) the SM time of all tiers fits 148 T.
static void plan_tiers(const std::vector<uint32_t>& cum, uint64_t n, uint32_t max_blocks, double total_blocks, int sm_count,
                       uint64_t warp_items[kMaxWarpCosched], uint64_t* pair_items, int force_c = 0) {
  for (int c = 0; c < kMaxWarpCosched; c++) warp_items[c] = 0;
  *pair_items = 0;
  const size_t nb = cum.size();
  std::vector<double> work_above(nb);  // blocks in bins > k
  double acc = 0;
  for (size_t k = nb; k-- > 0;) {
    work_above[k] = acc;
    const uint64_t cnt = (k == 0 ? n : cum[k - 1]) - cum[k];
    acc += (double)cnt * (double)(k + 1);
  }
  auto longer_than = [&](double thr, uint64_t* count, double* work) {  // items whose chain (bin + 1) exceeds thr
    if (thr < 1.0) {
      *count = n;
      *work = total_blocks;
      return;
    }
    const size_t k = std::min<size_t>((size_t)thr - 1, nb - 1);
    *count = cum[k];
    *work = work_above[k];
  };
  const double l1 = (double)max_blocks;
  const int c_first = force_c >= 1 && force_c <= kMaxWarpCosched ? force_c : 1;
  for (double T = l1 * kWarpChainRatio[c_first]; T < l1; T *= 1.01) {
    // class boundaries: an item with chain L runs c chains per scheduler iff L * ratio[c] <= T < L * ratio[c + 1]
    uint64_t k_above[kMaxWarpCosched + 2];  // [c] = items too long for warp class c + 1 (and every cheaper class)
    double w_above[kMaxWarpCosched + 2];
    k_above[0] = 0;
    w_above[0] = 0;
    for (int c = 1; c <= kMaxWarpCosched; c++) {
      const int next = c + 1;
      const double ratio = next <= kMaxWarpCosched ? kWarpChainRatio[next] : kPairChainRatio;
      longer_than(T / ratio, &k_above[c], &w_above[c]);
      if (force_c && c != force_c) {  // diagnostics: one warp class only
        k_above[c] = c < force_c ? 0 : k_above[force_c];
        w_above[c] = c < force_c ? 0 : w_above[force_c];
      }
    }
    uint64_t k_fast;
    double w_fast;
    longer_than(T, &k_fast, &w_fast);  // must not run one thread per item
    if (k_above[kMaxWarpCosched] == 0 && T < l1 * kPairChainRatio) continue;  // the pair tier alone cannot finish the longest in T
    uint64_t blocks = 0;
    double sm_time = 0;  // in units of (thread-tier permutation x SM)
    uint64_t cnt[kMaxWarpCosched];
    for (int c = 1; c <= kMaxWarpCosched; c++) {
      cnt[c - 1] = k_above[c] - k_above[c - 1];
      blocks += (cnt[c - 1] + 4 * c - 1) / (4 * c);
      sm_time += (w_above[c] - w_above[c - 1]) * kWarpChainRatio[c] / (4.0 * c);
    }
    const uint64_t k_p = k_fast - k_above[kMaxWarpCosched];
    blocks += (k_p + 63) / 64;
    sm_time += (w_fast - w_above[kMaxWarpCosched]) * kPairChainRatio / 64.0 + (total_blocks - w_fast) / 128.0;
    if (blocks + 1 > (uint64_t)sm_count) continue;
    if (sm_time > 0.95 * T * (double)sm_count) continue;
    // the thread-per-item tier gets the SMs the fast tiers leave (those stay busy for about T: their items are the
    // longest); its items are dispatched longest first, so it needs its share of SMs from the start
    if ((total_blocks - w_fast) / 128.0 > T * (double)((uint64_t)sm_count - blocks)) continue;
    for (int c = 0; c < kMaxWarpCosched; c++) warp_items[c] = cnt[c];
    *pair_items = k_p;
    return;
  }
}

// ---- small helpers of the launchers --------------------------------------------------------------------------------
// Calls f(std::integral_constant<int, L>()) for the L of Ls that equals `lanes` (a lane count known at run time picks the
// kernel instantiation) and returns its result; an unlisted value is CAPY_ERR_BAD_ARG.
template <int... Ls, class F>
static int with_lanes(int lanes, F&& f) {
  int rc = CAPY_ERR_BAD_ARG;
  (void)((lanes == Ls && ((rc = f(std::integral_constant<int, Ls>())), true)) || ...);
  return rc;
}

// a device buffer that is freed when it goes out of scope, unless release() hands it to a cache entry
struct CudaFree {
  void operator()(void* p) const { cudaFree(p); }
};
template <class T>
using DevPtr = std::unique_ptr<T, CudaFree>;
template <class T>
static cudaError_t dev_alloc(DevPtr<T>& p, size_t bytes) {
  T* q = nullptr;
  const cudaError_t e = cudaMalloc(&q, bytes);
  if (e == cudaSuccess) p.reset(q);
  return e;
}

// ---- plan of a ragged batch ----------------------------------------------------------------------------------------
// Length histogram of a batch in whole blocks of `stride_bytes` (bin kLenBins - 1 holds every longer item)
struct LenHist {
  uint64_t total_blocks = 0;  // sum of (bin + 1) over the items
  uint32_t max_bin = 0;       // largest non-empty bin
  uint32_t bins = 0;          // number of non-empty bins
  std::vector<uint32_t> cnt;  // items per bin when the histogram was taken on the host, else empty
};

// the histogram of a registered host offsets array
static void host_len_hist(const uint64_t* h_off, uint64_t n, uint32_t stride_bytes, LenHist* h) {
  h->cnt.assign(kLenBins, 0);
  const double inv = 1.0 / (double)stride_bytes;
  for (uint64_t i = 0; i < n; i++) {
    const uint64_t len = h_off[i + 1] - h_off[i];
    uint64_t q = (uint64_t)((double)len * inv);  // len / stride_bytes without a 64-bit division per item
    if (q * stride_bytes > len) q--;
    else if ((q + 1) * stride_bytes <= len) q++;
    const uint32_t b = q < kLenBins - 1 ? (uint32_t)q : kLenBins - 1;
    if (h->cnt[b]++ == 0) h->bins++;
    if (b > h->max_bin) h->max_bin = b;
    h->total_blocks += (uint64_t)b + 1;
  }
}

// Enqueues the device histogram and its scan, which leaves hist[k] = number of items in bins > k (the cursors of the
// scatter).  Without a host histogram the summary comes back to the host: a small copy and a stream synchronisation.
static int device_len_hist(capy_ctx* ctx, cudaStream_t st, const uint64_t* d_off, uint64_t n, uint32_t stride_bytes,
                           uint32_t* hist, LenHist* h) {
  uint32_t* summary = hist + kLenBins;
  CAPY_CUDA(ctx, cudaMemsetAsync(hist, 0, (size_t)kLenBins * 4 + 64, st));
  len_hist_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_off, n, stride_bytes, hist);
  len_scan_kernel<<<1, 1024, 0, st>>>(hist, summary);
  ctx->launches += 2;
  if (!h->cnt.empty()) return CAPY_OK;
  uint32_t h_sum[4];
  CAPY_CUDA(ctx, cudaMemcpyAsync(h_sum, summary, sizeof h_sum, cudaMemcpyDeviceToHost, st));
  CAPY_CUDA(ctx, cudaStreamSynchronize(st));
  h->total_blocks = (uint64_t)h_sum[0] | ((uint64_t)h_sum[1] << 32);
  h->max_bin = h_sum[2];
  h->bins = h_sum[3];
  return CAPY_OK;
}

// The plan a histogram gives: uniform block count, tiers of a chain-bound batch, occupancy throttle, and the scatter of
// the items into `order`, longest first (hist = the scanned device histogram).
static int plan_from_hist(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint64_t* d_off, uint64_t n,
                          uint32_t stride_bytes, const LenHist& h, uint32_t* hist, uint32_t* order, bool allow_pair,
                          int force_c, LaunchPlan* plan) {
  const uint32_t max_blocks = h.max_bin + 1;
  // time in units of one thread-per-state permutation on one scheduler: all work spread over every scheduler
  // (32 states per warp, one warp per scheduler) vs the longest chain
  const double ideal = (double)h.total_blocks / (32.0 * 4.0 * dc.sm_count);
  // Chain-bound batch: the longest items go to the warp-per-item and the two-threads-per-item tiers
  if (allow_pair && max_blocks > 64 && (double)max_blocks > 1.05 * ideal) {
    std::vector<uint32_t> cum(kLenBins);  // number of items in bins > k
    if (!h.cnt.empty()) {
      uint32_t above = 0;
      for (uint32_t k = kLenBins; k-- > 0;) {
        cum[k] = above;
        above += h.cnt[k];
      }
    } else {
      CAPY_CUDA(ctx, cudaMemcpyAsync(cum.data(), hist, (size_t)kLenBins * 4, cudaMemcpyDeviceToHost, st));
      CAPY_CUDA(ctx, cudaStreamSynchronize(st));
    }
    plan_tiers(cum, n, max_blocks, (double)h.total_blocks, dc.sm_count, plan->warp_items, &plan->pair_items, force_c);
  }
  if (h.bins == 1) plan->uniform_blocks = max_blocks;
  if (h.bins > 1) {  // (uniform lengths: nothing to order)
    len_scatter_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_off, n, stride_bytes, hist, order);
    ctx->launches++;
    CAPY_CUDA(ctx, cudaGetLastError());
    plan->order = order;
    plan->warps_per_smsp = 0;
    if ((double)max_blocks * 4.0 > 0.7 * ideal) {
      plan->warps_per_smsp = 3;
      if ((double)max_blocks * 3.0 > 0.7 * ideal) plan->warps_per_smsp = 2;
      if ((double)max_blocks * 2.0 > 0.7 * ideal) plan->warps_per_smsp = 1;
    }
  }
  return CAPY_OK;
}

// builds the descending-length order for a ragged batch; decides the occupancy throttle and how many of the
// longest items go to the warp-per-item and the two-threads-per-item tiers.
// The histogram comes back to the host (two small D2H copies + stream synchronisations) because the grid shape
// depends on it.  With the plan cache on (capy_gpu_set_plan_cache) the plan of an offsets array is kept, keyed by
// (device pointer, n, unit): every later call with the same array launches without touching the host, so the
// `_dev` entry points are fully asynchronous in steady state.
static int plan_ragged(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint64_t* d_off, uint64_t n,
                       uint32_t stride_bytes, LaunchPlan* plan, bool allow_pair = true, int force_c = 0) {
  *plan = LaunchPlan();
  if (n < 1 || n > 0xffffffffull) return CAPY_OK;
  // Host-buffer entry points: the offsets were staged from a host array that is still alive (HostChunk::in_packed registers it).
  // The lengths are read there, so nothing comes back from the device and the chunk pipeline of the host call never
  // waits for a stream.  Uniform lengths (the bulk case: fixed-size records) need no device work at all.
  const uint64_t* h_off = host_off_find(dc, d_off, n);
  LenHist h;
  if (h_off) {
    const uint64_t len0 = h_off[1] - h_off[0];
    bool uniform = true;
    for (uint64_t i = 1; i < n && uniform; i++) uniform = (h_off[i + 1] - h_off[i]) == len0;
    if (uniform) {  // nothing to order, no chain stands out
      plan->uniform_blocks = len0 / stride_bytes + 1;
      return CAPY_OK;
    }
    if (n > kHostPlanMaxItems) h_off = nullptr;  // a histogram of millions of items is cheaper on the device, round trip included
    else host_len_hist(h_off, n, stride_bytes, &h);
  }
  const bool cached = ctx->plan_cache.load() != 0 && force_c == 0 && !h_off;
  if (cached) {
    for (PlanEntry& e : dc.plans)
      if (e.off == d_off && e.n == n && e.unit == stride_bytes && e.allow_pair == allow_pair) {
        e.last_use = ++dc.use_clock;
        *plan = e.plan;
        return CAPY_OK;
      }
  }
  uint32_t* hist = (uint32_t*)scratch_get(dc, st, kPlanHist, (size_t)kLenBins * 4 + 64);
  DevPtr<uint32_t> owned;  // the order of a cached plan lives as long as its cache entry
  if (cached && dev_alloc(owned, (size_t)n * 4) != cudaSuccess) {
    cudaGetLastError();
    return CAPY_ERR_OOM;
  }
  uint32_t* order = cached ? owned.get() : (uint32_t*)scratch_get(dc, st, kPlanOrder, (size_t)n * 4);
  if (!hist || !order) return CAPY_ERR_OOM;
  int rc = device_len_hist(ctx, st, d_off, n, stride_bytes, hist, &h);
  if (rc) return rc;
  rc = plan_from_hist(ctx, dc, st, d_off, n, stride_bytes, h, hist, order, allow_pair, force_c, plan);
  if (rc) return rc;
  if (cached) {
    if (!plan->order) owned.reset();  // uniform batch: the entry records "nothing to do"
    if (dc.plans.size() >= kMaxPlanEntries) {  // evict the least recently used plan
      size_t lru = 0;
      for (size_t k = 1; k < dc.plans.size(); k++)
        if (dc.plans[k].last_use < dc.plans[lru].last_use) lru = k;
      if (dc.plans[lru].owned_order) cudaFree(dc.plans[lru].owned_order);  // waits for work that still reads it
      dc.plans.erase(dc.plans.begin() + lru);
    }
    PlanEntry e;
    e.off = d_off;
    e.n = n;
    e.unit = stride_bytes;
    e.allow_pair = allow_pair;
    e.plan = *plan;
    e.owned_order = owned.release();
    e.last_use = ++dc.use_clock;
    dc.plans.push_back(e);
  }
  return CAPY_OK;
}

// ---- one launch of a sponge job ------------------------------------------------------------------------------------
// The occupancy throttle of a plan: warps_per_smsp = W in 1..3 launches 128-thread blocks (one warp per scheduler) with
// a dynamic shared-memory footprint that lets W of them share an SM.
template <class Kernel>
static cudaError_t throttle(Kernel* kernel, const LaunchPlan& plan, unsigned* block, size_t* smem) {
  *smem = 0;
  if (plan.warps_per_smsp < 1 || plan.warps_per_smsp > 3) return cudaSuccess;
  *block = 128;
  *smem = (size_t)(227 * 1024 / plan.warps_per_smsp) - 1024;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
}

template <int LANES>
static int launch_sponge_t(capy_ctx* ctx, cudaStream_t stream, SpongeJob J, unsigned block, const LaunchPlan& plan) {
  if (plan.tiered()) {
    // chain-bound batch: warp blocks (one, two, three chains per scheduler), then pair blocks, then thread-per-item
    // blocks, one block per SM.  A block has 384 threads: a warp-tier block of class c uses 4 c warps, the other tiers
    // the first four; the rest exit at once.
    const uint64_t warp_items = plan.warp_items[0] + plan.warp_items[1] + plan.warp_items[2], pair_items = plan.pair_items;
    SpongeTiers tiers;
    uint32_t warp_blocks = 0;
    uint64_t rank = 0;
    for (int c = 0; c < 3; c++) {
      tiers.first_block[c] = warp_blocks;
      tiers.first_rank[c] = rank;
      warp_blocks += grid_for(plan.warp_items[c], 4 * (c + 1));
      rank += plan.warp_items[c];
    }
    tiers.warp_blocks = warp_blocks;
    tiers.pair_blocks = grid_for(2 * pair_items, 128);
    const unsigned solo_blocks = grid_for(J.n - pair_items - warp_items, 128);
    J.warp_items = warp_items;
    J.first = warp_items + pair_items;
    CAPY_CUDA(ctx, cudaFuncSetAttribute(sponge_tiered_kernel<LANES>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    sponge_tiered_kernel<LANES><<<warp_blocks + tiers.pair_blocks + solo_blocks, 384, 226 * 1024, stream>>>(J, tiers);
    ctx->launches++;
    CAPY_CUDA(ctx, cudaGetLastError());
    return CAPY_OK;
  }
  size_t smem;
  CAPY_CUDA(ctx, throttle(sponge_kernel<LANES>, plan, &block, &smem));
  sponge_kernel<LANES><<<grid_for(J.n, block), block, smem, stream>>>(J);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

// Block size for a one-thread-per-item kernel with few items: pick the block size whose block count
// spreads most evenly over the SMs (ties go to the larger block).
static unsigned pick_block(uint64_t n, int sm_count, int threads_per_sm) {
  unsigned best = 128;
  double best_eff = -1.0;
  for (unsigned bs : {128u, 64u, 32u}) {
    const uint64_t blocks = (n + bs - 1) / bs;
    const uint64_t slots = (uint64_t)sm_count * (threads_per_sm / bs);  // resident blocks per wave
    const uint64_t waves = (blocks + slots - 1) / slots;
    const double per_sm = (double)blocks / sm_count;
    const double busiest = waves > 1 ? (double)waves * (threads_per_sm / bs) : (double)((blocks + sm_count - 1) / sm_count);
    const double eff = per_sm / busiest;
    if (eff > best_eff + 0.02) {
      best_eff = eff;
      best = bs;
    }
  }
  return best;
}

// The kernels of a job are instantiated for the whole lanes of its rate: 21 for the 172-byte rate of D224 cSHAKE / KMAC
// (quirk Q7), rate / 8 for every other rate.
static int job_lanes(const SpongeJob& J) { return (int)(J.rate / 8); }

static int launch_sponge(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const SpongeJob& J, const LaunchPlan& plan) {
  if (J.n == 0) return CAPY_OK;
  const unsigned block = pick_block(J.n, dc.sm_count, 384);
  return with_lanes<9, 13, 17, 18, 19, 21>(job_lanes(J), [&](auto L) {
    return launch_sponge_t<decltype(L)::value>(ctx, stream, J, block, plan);
  });
}

// two jobs one after the other, both in the order of `plan`
static int launch_sponge_seq(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const SpongeJob& A, const SpongeJob& B,
                             const LaunchPlan& plan) {
  const int rc = launch_sponge(ctx, dc, stream, A, plan);
  if (rc) return rc;
  return launch_sponge(ctx, dc, stream, B, plan);
}

// ---- chain splitting of uniform batches (sponge.cuh: sponge_chain_kernel) --------------------------------------------
// Two dependent jobs in one launch need at least as many job-0 blocks as the GPU holds at once (CAPY_SPONGE_MINB per SM):
// a job-1 block of a smaller batch could wait for its job-0 block.  CAPY_NO_CHAIN_SPLIT turns them off (A/B switch for
// the probes).
static bool chain_jobs_fit(int sm_count, uint64_t n) {
  if (getenv("CAPY_NO_CHAIN_SPLIT") || sm_count < 1) return false;
  return (n + 127) / 128 >= (uint64_t)CAPY_SPONGE_MINB * (uint64_t)sm_count;
}

// Where to cut: the batch must fill the schedulers unevenly, be large enough for two dependent jobs (chain_jobs_fit), and
// leave the two halves about equally long; the cut lies inside -- or at the end of -- the absorb phase.  absorb_blocks
// counts the blocks after skip_blocks, squeeze_extra the permutations between squeeze blocks.  (A wrong estimate costs
// balance, never correctness: an item that is shorter than the cut simply has nothing left to absorb in job 1.)
static bool chain_cut(int sm_count, uint64_t n, uint64_t absorb_blocks, uint64_t squeeze_extra, uint64_t* cut) {
  if (!chain_jobs_fit(sm_count, n)) return false;
  const uint64_t warps = (n + 31) / 32, sched = 4ull * (uint64_t)sm_count;
  if (warps > 8 * sched) return false;
  auto fill = [&](uint64_t w) {
    const double x = (double)w / (double)sched;
    return x / std::ceil(x);
  };
  if (fill(2 * warps) < fill(warps) + 0.04) return false;
  const uint64_t perms = absorb_blocks + squeeze_extra;
  if (perms < 12) return false;
  uint64_t k = (perms + 1) / 2;
  if (k > absorb_blocks) k = absorb_blocks;
  if (3 * k < perms) return false;  // the absorb phase is too short to carry a half
  *cut = k;
  return true;
}

// two jobs over the same ranks in one launch, job 1 of an item after job 0 of that item (sponge_chain_kernel); with
// jobs = 1, J0 alone (and, with `resume`, as resumable streams)
static int launch_chain_jobs(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const SpongeJob& J0, const SpongeJob& J1,
                             bool data_dependent, uint32_t jobs = 2, const SpongeResume* resume = nullptr,
                             const SpongeSqueeze* squeeze = nullptr, const SpongeDual* dual = nullptr,
                             const SpongeCopy* copy = nullptr) {
  const uint32_t nb = (uint32_t)((J0.n + 127) / 128);
  uint32_t* sync = (uint32_t*)scratch_get(dc, stream, kChainSync, ((size_t)nb + 1) * sizeof(uint32_t));
  if (!sync) return CAPY_ERR_OOM;
  CAPY_CUDA(ctx, cudaMemsetAsync(sync, 0, ((size_t)nb + 1) * sizeof(uint32_t), stream));
  SpongeChain C;
  C.j[0] = J0;
  C.j[1] = J1;
  C.sync = sync;
  C.blocks_per_job = nb;
  C.data_dependent = data_dependent ? 1u : 0u;
  C.resume = resume ? *resume : SpongeResume{};
  C.squeeze = squeeze ? *squeeze : SpongeSqueeze{};
  C.dual = dual ? *dual : SpongeDual{};
  C.copy = copy ? *copy : SpongeCopy{};
  return with_lanes<9, 13, 17, 18, 19, 21>(job_lanes(J0), [&](auto L) {
    sponge_chain_kernel<decltype(L)::value><<<jobs * nb, 128, 0, stream>>>(C);
    ctx->launches++;
    CAPY_CUDA(ctx, cudaGetLastError());
    return CAPY_OK;
  });
}

// J (uniform batch, no order) as two dependent jobs cut after `cut` absorbed blocks
static int launch_sponge_chain(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const SpongeJob& J, uint64_t cut) {
  uint64_t* states = (uint64_t*)scratch_get(dc, stream, kChainStates, (size_t)J.n * 25 * sizeof(uint64_t));
  if (!states) return CAPY_ERR_OOM;
  SpongeJob J0 = J, J1 = J;
  J0.chain_out = states;
  J0.stop_block = J.skip_blocks + cut;
  J1.chain_in = states;
  J1.skip_blocks = (uint32_t)(J.skip_blocks + cut);
  return launch_chain_jobs(ctx, dc, stream, J0, J1, false);
}

// Whether a job is a uniform batch worth cutting along its chains, and where.  Uniform: a fixed-length job, or a plan
// that found one block count.  Jobs that write at per-item offsets or XOR into a buffer are not cut, nor are rates that
// are not lane-aligned (D224 cSHAKE / KMAC, quirk Q7).
static bool uniform_cut(const DeviceCtx& dc, const SpongeJob& J, const LaunchPlan& plan, uint64_t* cut) {
  if (J.out_off || J.xor_in || plan.order || (J.rate & 7u) != 0) return false;
  const uint64_t msg_blocks = J.off ? plan.uniform_blocks : J.msg_len / J.rate + 1;  // the last one holds the trailer
  if (!msg_blocks) return false;
  // blocks absorbed after skip_blocks: the rest of the prefix, the key block bytepad(encode_string(K), w), the message
  uint64_t absorb = msg_blocks;
  if (J.keys) absorb += ((uint64_t)J.key_len + 8) / J.w + 1;
  if (!J.skip_blocks) absorb += J.prefix_len / J.rate;
  const uint64_t sq = 8ull * J.sq_lanes, squeeze_extra = J.out_bytes ? (J.out_bytes + sq - 1) / sq - 1 : 0;
  return chain_cut(dc.sm_count, J.n, absorb, squeeze_extra, cut);
}

// Launches a built job in the order of `plan`: a uniform batch as two dependent jobs when uniform_cut says so, anything
// else as one launch.
static int run_sponge(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, SpongeJob J, const LaunchPlan& plan) {
  J.order = plan.order;
  uint64_t cut;
  if (uniform_cut(dc, J, plan, &cut)) return launch_sponge_chain(ctx, dc, stream, J, cut);
  return launch_sponge(ctx, dc, stream, J, plan);
}

// ---- the operators: rate, squeeze width, trailer and pad of each; callers add their data and output fields ------------
static SpongeJob sha3_job(int d) {
  SpongeJob J{};
  J.trailer_len = 1;
  J.sha3_suffix = 1;  // 06 | 86 from the message length (Q2)
  J.rate = sha3_rate(d);
  J.sq_lanes = squeeze_lanes(d);  // the first d/8 bytes are all that is kept
  return J;
}

// q4: N = S = "" (quirk Q4, shake_functions.rs:59-61)
static SpongeJob cshake_job(int d, bool q4) {
  SpongeJob J{};
  J.trailer = 0x04;  // shake_functions.rs:57
  J.trailer_len = 1;
  if (q4) J.q4_rate = sha3_rate(d);
  J.rate = cshake_rate(d);
  J.sq_lanes = squeeze_lanes(d);
  return J;
}

// on top of J, the caller's per-item fields
static SpongeJob kmac_job(int d, SpongeJob J = SpongeJob{}) {
  J.trailer = 0x040100u;  // right_encode(0) = 00 01 (shake_functions.rs:86) then 04 (:57)
  J.trailer_len = 3;
  J.rate = cshake_rate(d);
  J.sq_lanes = squeeze_lanes(d);
  return J;
}

static SpongeJob shake_job(int shake_bits) {
  SpongeJob J{};
  J.trailer = 0x1F;
  J.trailer_len = 1;
  J.fips_pad = 1;
  J.rate = shake_rate(shake_bits);
  J.sq_lanes = squeeze_lanes(2 * shake_bits);
  return J;
}

// the cached prefix P of a cSHAKE / KMAC job (get_prefix); its bytepad width is the rate
static void set_prefix(SpongeJob& J, const PrefixState* ps) {
  J.prefix = ps->d_prefix;
  J.prefix_len = ps->prefix_len;
  J.init_state = ps->skip_blocks ? ps->d_state : nullptr;
  J.skip_blocks = ps->skip_blocks;
  J.w = J.rate;
}

// ---- SHA3-d ------------------------------------------------------------------------------------
// tail_readable: the 8-byte word that holds the last message byte of the LAST row may be read in full (the host entry
// points stage into buffers with slack; a caller-owned device buffer may end with the last message byte)
static int launch_sha3(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, int d, const uint8_t* data, const uint64_t* off,
                       uint64_t msg_len, uint64_t stride, uint64_t n, uint8_t* out, uint32_t flags = 0,
                       bool tail_readable = true) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  if (!off && !tail_readable && (msg_len & 7u) != 0 && n > 1 && (reinterpret_cast<uintptr_t>(data) & 7u) == 0 &&
      (stride & 7u) == 0 && (reinterpret_cast<uintptr_t>(out) & 3u) == 0) {
    // every row but the last has its tail word inside its own stride or the next row; the last row goes through the
    // byte-granular kernel, which never reads past the message
    int rc = launch_sha3(ctx, dc, stream, d, data, nullptr, msg_len, stride, n - 1, out, flags, true);
    if (rc) return rc;
    return launch_sha3(ctx, dc, stream, d, data + (n - 1) * stride, nullptr, msg_len, stride, 1, out + (n - 1) * (uint64_t)(d / 8),
                       flags, false);
  }
  SpongeJob J = sha3_job(d);
  if (!off && (reinterpret_cast<uintptr_t>(data) & 15u) == 0 && (reinterpret_cast<uintptr_t>(out) & 15u) == 0 &&
      (stride & 15u) == 0 && (d == 256 || d == 512) && msg_len >= 16 && (msg_len & 15u) == 0 && msg_len < J.rate) {
    // compile-time block layout: single-block messages of a whole number of 16-byte rows (cfg 1 is 64 B at D256)
    const unsigned block = 128, grid = grid_for(n, block);
    const uint4* dq = reinterpret_cast<const uint4*>(data);
    uint4* oq = reinterpret_cast<uint4*>(out);
    const uint64_t s16 = stride / 16;
    const int msg_lanes = (int)(msg_len / 8);  // 2, 4, .. 16 at D256; 2, 4, 6, 8 at D512
    const int rc = d == 256 ? with_lanes<2, 4, 6, 8, 10, 12, 14, 16>(msg_lanes, [&](auto M) {
      sha3_short_kernel<17, decltype(M)::value><<<grid, block, 0, stream>>>(dq, s16, 0x06u, oq, 32, n);
      return CAPY_OK;
    }) : with_lanes<2, 4, 6, 8>(msg_lanes, [&](auto M) {
      sha3_short_kernel<9, decltype(M)::value><<<grid, block, 0, stream>>>(dq, s16, 0x06u, oq, 64, n);
      return CAPY_OK;
    });
    if (rc) return rc;
    ctx->launches++;
    CAPY_CUDA(ctx, cudaGetLastError());
    return CAPY_OK;
  }
  J.data = data;
  J.off = off;
  J.msg_len = msg_len;
  J.msg_stride = stride;
  J.out = out;
  J.out_stride = J.out_bytes = (uint64_t)d / 8;
  J.n = n;
  // long equal messages that fill the GPU unevenly are cut along the chains (run_sponge), which the uniform kernel cannot
  // do; the uniform kernel stores 4-byte granules (28- and 48-byte digests) and reads whole 8-byte words
  uint64_t cut;
  if (!off && !uniform_cut(dc, J, LaunchPlan(), &cut) && (reinterpret_cast<uintptr_t>(data) & 7u) == 0 &&
      (stride & 7u) == 0 && (reinterpret_cast<uintptr_t>(out) & 3u) == 0 && (tail_readable || (msg_len & 7u) == 0)) {
    const uint32_t suffix = (msg_len % 136u == 135u) ? 0x86u : 0x06u;  // shake_functions.rs:25-29 (Q2)
    const unsigned block = 128, grid = grid_for(n, block);
    return with_lanes<9, 13, 17, 18>(job_lanes(J), [&](auto L) {
      sha3_uniform_kernel<decltype(L)::value><<<grid, block, 0, stream>>>(data, stride, msg_len, suffix, out, d / 8, n);
      ctx->launches++;
      CAPY_CUDA(ctx, cudaGetLastError());
      return CAPY_OK;
    });
  }
  LaunchPlan plan;
  if (off && !(flags & CAPY_FLAG_NO_SORT)) {
    int rc = plan_ragged(ctx, dc, stream, off, n, J.rate, &plan, !(flags & CAPY_FLAG_NO_PAIR),
                         (int)((flags >> CAPY_FLAG_WARP_COSCHED_SHIFT) & 3u));
    if (rc) return rc;
  }
  return run_sponge(ctx, dc, stream, J, plan);
}

// ---- cSHAKE / KMAC prefix -----------------------------------------------------------------------
static void host_left_encode(std::string& o, uint64_t v) {  // aux_functions.rs:34-49
  if (v == 0) {
    o.push_back(1);
    o.push_back(0);
    return;
  }
  int nb = 8;
  while (nb > 1 && ((v >> (8 * (nb - 1))) & 0xFF) == 0) nb--;
  o.push_back((char)nb);
  for (int i = nb - 1; i >= 0; i--) o.push_back((char)((v >> (8 * i)) & 0xFF));
}
static void host_encode_string(std::string& o, const uint8_t* s, size_t n) {  // aux_functions.rs:24-28
  host_left_encode(o, (uint64_t)n * 8);
  o.append(reinterpret_cast<const char*>(s), n);
}

static int get_prefix(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, int d, const uint8_t* fn, uint32_t fn_len,
                      const uint8_t* cs, uint32_t cs_len, PrefixState** out) {
  std::string key;
  key.push_back((char)(d >> 8));
  key.push_back((char)d);
  host_left_encode(key, fn_len);
  key.append(reinterpret_cast<const char*>(fn), fn_len);
  key.append(reinterpret_cast<const char*>(cs), cs_len);
  auto it = dc.prefix_cache.find(key);
  if (it != dc.prefix_cache.end()) {
    it->second.last_use = ++dc.use_clock;
    *out = &it->second;
    return CAPY_OK;
  }
  // The customisation string is caller-controlled (compute_tagged_hash's S): bound the cache, least recently used out.
  // cudaFree waits for work that still reads the evicted buffers.
  if (dc.prefix_cache.size() >= kMaxPrefixEntries) {
    auto lru = dc.prefix_cache.begin();
    for (auto k = dc.prefix_cache.begin(); k != dc.prefix_cache.end(); ++k)
      if (k->second.last_use < lru->second.last_use) lru = k;
    if (lru->second.d_state) cudaFree(lru->second.d_state);
    if (lru->second.d_prefix) cudaFree(lru->second.d_prefix);
    dc.prefix_cache.erase(lru);
  }
  const uint32_t w = cshake_rate(d);  // the bytepad width
  std::string p;  // bytepad(encode_string(N) || encode_string(S), w)   shake_functions.rs:50-55
  host_left_encode(p, w);
  host_encode_string(p, fn, fn_len);
  host_encode_string(p, cs, cs_len);
  p.append(w - p.size() % w, '\0');  // aux_functions.rs:14-16 (quirk Q3)
  PrefixState ps;
  ps.prefix_len = (uint32_t)p.size();
  DevPtr<uint8_t> d_prefix;  // nothing is cached on failure: these free what was allocated
  DevPtr<uint64_t> d_state;
  CAPY_CUDA(ctx, dev_alloc(d_prefix, p.size()));
  CAPY_CUDA(ctx, dev_alloc(d_state, 25 * sizeof(uint64_t)));
  CAPY_CUDA(ctx, cudaMemcpyAsync(d_prefix.get(), p.data(), p.size(), cudaMemcpyHostToDevice, stream));
  if (w % 8 == 0) {
    // the prefix is a whole number of blocks: fold it into a cached state once
    ps.skip_blocks = ps.prefix_len / w;
    const int rc = with_lanes<17, 19, 21>((int)(w / 8), [&](auto L) {
      prefix_state_kernel<decltype(L)::value><<<1, 32, 0, stream>>>(d_prefix.get(), ps.skip_blocks, d_state.get());
      ctx->launches++;
      CAPY_CUDA(ctx, cudaGetLastError());
      return CAPY_OK;
    });
    if (rc) return rc;
  } else {
    ps.skip_blocks = 0;  // D224: w = 172 is not lane aligned (quirk Q7), blocks straddle the prefix end
  }
  // the host string dies at return, and later calls may use the entry from other streams: wait for the build
  CAPY_CUDA(ctx, cudaStreamSynchronize(stream));
  ps.d_prefix = d_prefix.release();
  ps.d_state = d_state.release();
  ps.last_use = ++dc.use_clock;
  auto ins = dc.prefix_cache.emplace(key, ps);
  *out = &ins.first->second;
  return CAPY_OK;
}

static int launch_cshake(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, int d, const uint8_t* data,
                         const uint64_t* off, uint64_t n, const uint8_t* fn, uint32_t fn_len, const uint8_t* cs,
                         uint32_t cs_len, uint64_t out_bits, uint8_t* out) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0 || out_bits / 8 == 0) return CAPY_OK;
  PrefixState* ps;
  int rc = get_prefix(ctx, dc, stream, d, fn, fn_len, cs, cs_len, &ps);
  if (rc) return rc;
  SpongeJob J = cshake_job(d, fn_len == 0 && cs_len == 0);
  set_prefix(J, ps);
  J.data = data;
  J.off = off;
  J.out = out;
  J.out_stride = J.out_bytes = out_bits / 8;
  J.n = n;
  LaunchPlan plan;
  rc = plan_ragged(ctx, dc, stream, off, n, J.rate & ~7u, &plan);
  if (rc) return rc;
  return run_sponge(ctx, dc, stream, J, plan);
}

// the pass's own per-item fields, with the KMAC operator fields and the prefix of (d, custom)
static int build_kmac_job(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& a, SpongeJob* out) {
  static const uint8_t kKmac[4] = {'K', 'M', 'A', 'C'};
  PrefixState* ps;
  int rc = get_prefix(ctx, dc, stream, a.d_bits, kKmac, 4, reinterpret_cast<const uint8_t*>(a.custom.data()),
                      (uint32_t)a.custom.size(), &ps);
  if (rc) return rc;
  SpongeJob J = kmac_job(a.d_bits, a.job);
  set_prefix(J, ps);
  if (!J.data) J.data = J.keys;  // no message: never read, but the kernels still offset it per item
  *out = J;
  return CAPY_OK;
}

static int plan_kmac(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& a, const SpongeJob& J, LaunchPlan* plan) {
  *plan = LaunchPlan();
  if (a.no_sort) return CAPY_OK;
  if (J.off) return plan_ragged(ctx, dc, stream, J.off, J.n, J.rate & ~7u, plan);
  // keystream shape (sha3/encryptable.rs:41): the work of an item is its squeeze length
  if (J.out_off) return plan_ragged(ctx, dc, stream, J.out_off, J.n, 8u * J.sq_lanes, plan);
  return CAPY_OK;
}

int launch_kmac_xof(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& a) {
  if (!valid_secparam(a.d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (a.job.n == 0) return CAPY_OK;
  if (!a.job.out_off && a.job.out_bytes == 0) return CAPY_OK;
  SpongeJob J;
  int rc = build_kmac_job(ctx, dc, stream, a, &J);
  if (rc) return rc;
  LaunchPlan plan;
  rc = plan_kmac(ctx, dc, stream, a, J, &plan);
  if (rc) return rc;
  return run_sponge(ctx, dc, stream, J, plan);
}

// Two independent KMACXOF passes over the same items (same d, same n) as ONE launch: warps alternate between the two
// jobs, so a batch whose single pass fills the schedulers unevenly (2^16 items = 3.46 warps per scheduler, the last
// wave 15 % full) runs as 6.92 warps per scheduler.  The authenticated-encryption seal is such a pair: the tag pass
// absorbs the message, the keystream pass squeezes into the XOR (sha3/encryptable.rs:36-42).  Both jobs follow the
// plan of `a`.  Chain-bound batches (tiers) run the two passes one after the other.
template <int LANES>
static int launch_sponge2_t(capy_ctx* ctx, cudaStream_t stream, const SpongeJob& A, const SpongeJob& B, unsigned block,
                            const LaunchPlan& plan) {
  SpongeJob2 JJ;
  JJ.j[0] = A;
  JJ.j[1] = B;
  size_t smem;
  CAPY_CUDA(ctx, throttle(sponge_kernel2<LANES>, plan, &block, &smem));
  const uint64_t warps = 2 * ((A.n + 31) / 32);
  sponge_kernel2<LANES><<<grid_for(warps * 32, block), block, smem, stream>>>(JJ);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

int launch_kmac_xof2(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& a, const KmacPass& b) {
  if (!valid_secparam(a.d_bits) || a.d_bits != b.d_bits || a.job.n != b.job.n) return CAPY_ERR_BAD_ARG;
  if (a.job.n == 0) return CAPY_OK;
  SpongeJob JA, JB;
  int rc = build_kmac_job(ctx, dc, stream, a, &JA);
  if (rc) return rc;
  rc = build_kmac_job(ctx, dc, stream, b, &JB);
  if (rc) return rc;
  LaunchPlan plan;
  rc = plan_kmac(ctx, dc, stream, a, JA, &plan);
  if (rc) return rc;
  JA.order = JB.order = plan.order;
  if (plan.tiered()) return launch_sponge_seq(ctx, dc, stream, JA, JB, plan);
  const unsigned block = pick_block(2 * JA.n, dc.sm_count, 384);
  return with_lanes<17, 19, 21>(job_lanes(JA), [&](auto L) {
    return launch_sponge2_t<decltype(L)::value>(ctx, stream, JA, JB, block, plan);
  });
}

// Two KMACXOF passes where the SECOND absorbs what the FIRST wrote for the same item (authenticated decryption: the
// keystream pass recovers the plaintext, the tag pass runs over it -- sha3/encryptable.rs:66-75): one launch of
// dependent jobs instead of two kernels, so the partial wave of the first pass is filled by the second.  Both follow the
// plan (work order) of `second`.  Small or chain-bound batches run the two passes one after the other.
int launch_kmac_xof_dep(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& first, const KmacPass& second) {
  if (!valid_secparam(first.d_bits) || first.d_bits != second.d_bits || first.job.n != second.job.n) return CAPY_ERR_BAD_ARG;
  if (first.job.n == 0) return CAPY_OK;
  SpongeJob J0, J1;
  int rc = build_kmac_job(ctx, dc, stream, first, &J0);
  if (rc) return rc;
  rc = build_kmac_job(ctx, dc, stream, second, &J1);
  if (rc) return rc;
  LaunchPlan plan;
  rc = plan_kmac(ctx, dc, stream, second, J1, &plan);
  if (rc) return rc;
  J0.order = J1.order = plan.order;
  if (plan.tiered() || (J0.rate & 7u) != 0 || !chain_jobs_fit(dc.sm_count, J0.n))
    return launch_sponge_seq(ctx, dc, stream, J0, J1, plan);
  return launch_chain_jobs(ctx, dc, stream, J0, J1, true);
}

// ---- resumable streams (capy_hasher) -------------------------------------------------------------------------------
// Every update and final is ONE single-job launch of sponge_chain_kernel over a range of the hasher's items on one device
// (thread per item, no order, no cut); SpongeJob::carry switches sponge_item to the resumed stream.
static int hasher_check(const capy_ctx* ctx, const capy_hasher* h) { return h && ctx && h->ctx == ctx ? CAPY_OK : CAPY_ERR_BAD_ARG; }
static uint64_t hasher_items(const capy_hasher* h, int k) { return h->first[k + 1] - h->first[k]; }
static bool hasher_any_finished(const capy_hasher* h) {
  for (char f : h->finished)
    if (f) return true;
  return false;
}
// a stream of `kind` in `pass` on device k, not finished
static bool hasher_dev_in_pass(const capy_hasher* h, int k, int kind, int pass) {
  return h->kind == kind && !h->finished[k] && h->pass[k] == pass;
}
static bool hasher_in_pass(const capy_hasher* h, int kind, int pass) {
  for (size_t k = 0; k < h->finished.size(); k++)
    if (!hasher_dev_in_pass(h, (int)k, kind, pass)) return false;
  return true;
}
std::vector<Range> hasher_shards(const capy_hasher* h) {
  std::vector<Range> s;
  for (size_t k = 0; k + 1 < h->first.size(); k++) s.push_back({h->first[k], h->first[k + 1]});
  return s;
}

// the outputs capy_hasher_final takes: SHA3-d digests, any KMACXOF output, the tag of encryption streams; verification
// streams end in capy_hasher_verify_final
static bool hasher_final_fits(const capy_hasher* h, uint64_t out_bits, const uint64_t* out_off) {
  switch (h->kind) {
    case kSha3Stream: return out_bits == (uint64_t)h->d_bits && !out_off;
    case kKmacStream: return true;
    case kEncryptStream: return out_bits == h->tag_bits && !out_off;
    default: return false;
  }
}

// the operator of the hasher's streams; its prefix and keys are already in their states
static SpongeJob hasher_operator(const capy_hasher* h) { return h->kmac ? kmac_job(h->d_bits) : sha3_job(h->d_bits); }

// the job of an update or a final over the items [j0, j0 + n) of device k (indices on that device), and its streams
static SpongeJob hasher_job(const capy_hasher* h, int k, uint64_t j0, uint64_t n, SpongeResume* R) {
  SpongeJob J = hasher_operator(h);
  J.chain_in = h->d_state[k] + j0;
  J.n = n;
  R->carry = h->d_carry[k] + j0 * h->rate;
  R->totals = h->d_total[k] + j0;
  R->state_n = hasher_items(h, k);
  return J;
}

static int hasher_update_items(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, capy_hasher* h, uint64_t j0, uint64_t n,
                               const uint8_t* d_data, const uint64_t* d_off) {
  if (n == 0) return CAPY_OK;
  SpongeResume R;
  SpongeJob J = hasher_job(h, dc.index, j0, n, &R);
  J.chain_out = h->d_state[dc.index] + j0;
  J.stop_block = ~0ull;
  J.data = d_data;
  J.off = d_off;
  return launch_chain_jobs(ctx, dc, st, J, J, false, 1, &R);
}

// an update of encryption streams: job 0 absorbs the plaintext into the tag streams, job 1 XORs the keystream into it.
// Job 1 of a block starts after job 0 of that block, so the tag has read the plaintext when `ct == data` overwrites it.
static int hasher_encrypt_items(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, capy_hasher* h, uint64_t j0, uint64_t n,
                                const uint8_t* d_data, const uint64_t* d_off, uint8_t* d_ct) {
  if (n == 0) return CAPY_OK;
  const int k = dc.index;
  SpongeResume R;
  SpongeJob J0 = hasher_job(h, k, j0, n, &R);
  J0.chain_out = h->d_state[k] + j0;
  J0.stop_block = ~0ull;
  J0.data = d_data;
  J0.off = d_off;
  SpongeJob J1 = hasher_operator(h);
  J1.chain_in = J1.chain_out = h->d_ks_state[k] + j0;
  J1.data = d_data;
  J1.off = d_off;
  J1.out = d_ct;
  J1.n = n;
  const SpongeSqueeze S{h->d_ks_pos[k] + j0, hasher_items(h, k)};
  return launch_chain_jobs(ctx, dc, st, J0, J1, false, 2, &R, &S);
}

// an update of sign streams in pass 2 (A: the "T" stream, B: the second "N" stream) or of decryption streams (A: the
// keystream, B: the tag stream; d_out in pass 2 only): one launch of the two-state path
static int hasher_dual_items(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, capy_hasher* h, uint64_t j0, uint64_t n,
                             const uint8_t* d_data, const uint64_t* d_off, uint8_t* d_out) {
  if (n == 0) return CAPY_OK;
  const int k = dc.index;
  SpongeResume R;
  SpongeJob J = hasher_job(h, k, j0, n, &R);
  SpongeDual D{};
  if (h->kind == kDecryptStream) {
    J.chain_out = h->d_ks_state[k] + j0;
    D.b_state = h->d_state[k] + j0;
    D.open = 1;
    D.out = d_out;
    D.verdict = h->d_verdict[k] + j0;
  } else {
    J.chain_out = h->d_state[k] + j0;
    D.b_state = h->d_state2[k] + j0;
  }
  J.chain_in = J.chain_out;
  J.stop_block = ~0ull;
  J.data = d_data;
  J.off = d_off;
  return launch_chain_jobs(ctx, dc, st, J, J, false, 1, &R, nullptr, &D);
}

// a piece of every stream: pass 1 of sign streams is a plain KMAC stream update, pass 2 and decryption streams run two
// states
static int hasher_piece_items(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, capy_hasher* h, uint64_t j0, uint64_t n,
                              const uint8_t* d_data, const uint64_t* d_off) {
  if (h->kind == kDecryptStream || (h->kind == kSignStream && h->pass[dc.index] == 2))
    return hasher_dual_items(ctx, dc, st, h, j0, n, d_data, d_off, nullptr);
  return hasher_update_items(ctx, dc, st, h, j0, n, d_data, d_off);
}

int hasher_final_items(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const capy_hasher* h, uint64_t j0, uint64_t n,
                       uint64_t out_bytes, const uint64_t* d_out_off, uint8_t* d_out, const uint64_t* state) {
  if (n == 0 || (!d_out_off && out_bytes == 0)) return CAPY_OK;
  SpongeResume R;
  SpongeJob J = hasher_job(h, dc.index, j0, n, &R);
  if (state) J.chain_in = state + j0;
  J.out = d_out;
  J.out_off = d_out_off;
  J.out_stride = J.out_bytes = out_bytes;
  return launch_chain_jobs(ctx, dc, st, J, J, false, 1, &R);
}

// the final of verification streams: h' through the tag final, then ok = (h' == h) && !bad
static int hasher_verify_items(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const capy_hasher* h, uint64_t j0, uint64_t n,
                               uint8_t* d_ok, int* d_bad_flag) {
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(hp, uint8_t, kEdTmp56B, n * 56);
  const int rc = hasher_final_items(ctx, dc, st, h, j0, n, 56, nullptr, hp);
  if (rc) return rc;
  return launch_verify_compare(ctx, st, hp, h->d_h[dc.index] + 56 * j0, h->d_bad[dc.index] + j0, d_ok, d_bad_flag, n);
}

int launch_kmac_state(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& a, bool trailer, uint64_t* states) {
  SpongeJob J;
  const int rc = build_kmac_job(ctx, dc, stream, a, &J);
  if (rc) return rc;
  if (!trailer) {
    J.trailer = 0;
    J.trailer_len = 0;
  }
  J.chain_out = states;
  J.stop_block = ~0ull;
  return launch_chain_jobs(ctx, dc, stream, J, J, false, 1);
}

int hasher_restart(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, capy_hasher* h) {
  const size_t m = (size_t)hasher_items(h, dc.index);
  CAPY_CUDA(ctx, cudaMemsetAsync(h->d_carry[dc.index], 0, m * h->rate, st));
  CAPY_CUDA(ctx, cudaMemsetAsync(h->d_total[dc.index], 0, m * 8, st));
  return CAPY_OK;
}

// Items are dealt out in equal contiguous ranges.
int hasher_create(capy_ctx* ctx, int d_bits, int kind, uint64_t n, capy_hasher** out, uint32_t tag_bits) {
  capy_hasher* h = new (std::nothrow) capy_hasher();
  if (!h) return CAPY_ERR_OOM;
  h->ctx = ctx;
  h->d_bits = d_bits;
  h->kind = kind;
  h->kmac = kind != kSha3Stream;
  h->tag_bits = tag_bits;
  h->rate = hasher_operator(h).rate;
  h->n = n;
  const uint64_t nd = ctx->devs.size();
  for (uint64_t k = 0; k <= nd; k++) h->first.push_back((n / nd) * k + std::min(k, n % nd));
  for (const DeviceCtx& dc : ctx->devs) h->dev.push_back(dc.dev);
  h->d_state.assign(nd, nullptr);
  h->d_carry.assign(nd, nullptr);
  h->d_total.assign(nd, nullptr);
  h->d_ks_state.assign(nd, nullptr);
  h->d_ks_pos.assign(nd, nullptr);
  h->d_h.assign(nd, nullptr);
  h->d_bad.assign(nd, nullptr);
  h->d_state2.assign(nd, nullptr);
  h->d_s.assign(nd, nullptr);
  h->d_k.assign(nd, nullptr);
  h->d_s_be.assign(nd, nullptr);
  h->d_n1.assign(nd, nullptr);
  h->d_state0.assign(nd, nullptr);
  h->d_ks_state0.assign(nd, nullptr);
  h->d_verdict.assign(nd, nullptr);
  h->pass.assign(nd, kind == kSignStream || kind == kDecryptStream ? 1 : 0);
  h->finished.assign(nd, 0);
  for (DeviceCtx& dc : ctx->devs) {
    const uint64_t m = hasher_items(h, dc.index);
    if (m == 0) continue;
    std::lock_guard<std::mutex> lk(*dc.mu);
    DeviceGuard g(dc.dev);
    const cudaStream_t st = dc.streams[0];
    const int rc = [&]() -> int {
      auto zeroed = [&](auto*& p, size_t bytes) -> int {
        CAPY_CUDA(ctx, cudaMalloc(&p, bytes));
        CAPY_CUDA(ctx, cudaMemsetAsync(p, 0, bytes, st));
        return CAPY_OK;
      };
      const int k = dc.index;
      int r = zeroed(h->d_state[k], (size_t)m * 200);
      if (!r) r = zeroed(h->d_carry[k], (size_t)m * h->rate);
      if (!r) r = zeroed(h->d_total[k], (size_t)m * 8);
      const bool sign = kind == kSignStream, dec = kind == kDecryptStream;
      if (!r && (kind == kEncryptStream || dec)) r = zeroed(h->d_ks_state[k], (size_t)m * 200);
      if (!r && kind == kEncryptStream) r = zeroed(h->d_ks_pos[k], (size_t)m * 8);
      if (!r && kind == kVerifyStream) r = zeroed(h->d_h[k], (size_t)m * 56);
      if (!r && kind == kVerifyStream) r = zeroed(h->d_bad[k], (size_t)m);
      if (!r && sign) r = zeroed(h->d_state2[k], (size_t)m * 200);
      if (!r && sign) r = zeroed(h->d_s[k], (size_t)m * 56);
      if (!r && sign) r = zeroed(h->d_k[k], (size_t)m * 56);
      if (!r && sign) r = zeroed(h->d_s_be[k], (size_t)m * 56);
      if (!r && sign) r = zeroed(h->d_n1[k], (size_t)m * 56);
      if (!r && dec) r = zeroed(h->d_state0[k], (size_t)m * 200);
      if (!r && dec) r = zeroed(h->d_ks_state0[k], (size_t)m * 200);
      if (!r && dec) r = zeroed(h->d_h[k], (size_t)m * (tag_bits / 8));
      if (!r && dec) r = zeroed(h->d_verdict[k], (size_t)m);
      if (!r && dec && tag_bits == 448) r = zeroed(h->d_bad[k], (size_t)m);
      if (r) return r;
      CAPY_CUDA(ctx, cudaStreamSynchronize(st));
      return CAPY_OK;
    }();
    if (rc) {
      cudaGetLastError();
      capy_hasher_free(h);
      return rc;
    }
  }
  *out = h;
  return CAPY_OK;
}

// ---- checkpoints and forks of SHA3-d / KMACXOF streams (capy_hasher_export / _import / _fork) -------------------------
// The blob format is decided here alone; capy_gpu.h documents it.  Header (64 bytes, little-endian): "CAPYHSTR", u32
// version, u32 kind (0 SHA3-d, 1 KMACXOF), u32 d_bits, u32 rate, u32 record bytes, u32 zero, u64 n, zeros; then n records
// of 208 + rate bytes (SpongeCopy).  Every copy is one launch of the copy path of sponge_chain_kernel.
constexpr uint64_t kBlobHeader = 64;
constexpr uint32_t kBlobVersion = 1;
static const char kBlobMagic[8] = {'C', 'A', 'P', 'Y', 'H', 'S', 'T', 'R'};

static uint64_t blob_record(uint32_t rate) { return 208ull + rate; }
// the kinds a blob can hold, and only while no device has finished its items
static bool hasher_portable(const capy_hasher* h) {
  return (h->kind == kSha3Stream || h->kind == kKmacStream) && !hasher_any_finished(h);
}
static uint64_t get_le(const uint8_t* p, int bytes) {
  uint64_t v = 0;
  for (int k = bytes - 1; k >= 0; k--) v = (v << 8) | p[k];
  return v;
}
static void put_le(uint8_t* p, uint64_t v, int bytes) {
  for (int k = 0; k < bytes; k++) p[k] = (uint8_t)(v >> (8 * k));
}

struct BlobHeader {
  int kind;  // kSha3Stream or kKmacStream
  int d_bits;
  uint32_t rate;
  uint64_t n;
};
static int blob_parse(const uint8_t* blob, uint64_t blob_len, BlobHeader* b) {
  if (!blob || blob_len < kBlobHeader || memcmp(blob, kBlobMagic, 8) != 0) return CAPY_ERR_BAD_ARG;
  const uint32_t version = (uint32_t)get_le(blob + 8, 4), kind = (uint32_t)get_le(blob + 12, 4);
  const int d = (int)get_le(blob + 16, 4);
  const uint32_t rate = (uint32_t)get_le(blob + 20, 4), rec = (uint32_t)get_le(blob + 24, 4);
  if (version != kBlobVersion || kind > 1 || !valid_secparam(d) || (kind == 1 && d == 224)) return CAPY_ERR_BAD_ARG;
  const uint32_t want = kind == 1 ? cshake_rate(d) : sha3_rate(d);
  if (rate != want || rec != blob_record(rate) || get_le(blob + 28, 4) != 0) return CAPY_ERR_BAD_ARG;
  for (uint64_t k = 40; k < kBlobHeader; k++)
    if (blob[k]) return CAPY_ERR_BAD_ARG;
  const uint64_t n = get_le(blob + 32, 8);
  if (n > (blob_len - kBlobHeader) / rec || blob_len - kBlobHeader != n * rec) return CAPY_ERR_BAD_ARG;
  b->kind = kind == 1 ? kKmacStream : kSha3Stream;
  b->d_bits = d;
  b->rate = rate;
  b->n = n;
  return CAPY_OK;
}

// the streams of device k from item j0 on (indices on that device), as a side of a copy
static SpongeStreams hasher_side(const capy_hasher* h, int k, uint64_t j0) {
  SpongeStreams s{};
  s.state = h->d_state[k] + j0;
  s.carry = h->d_carry[k] + j0 * h->rate;
  s.totals = h->d_total[k] + j0;
  s.state_n = hasher_items(h, k);
  return s;
}
static SpongeStreams record_side(uint8_t* rec) {
  SpongeStreams s{};
  s.rec = rec;
  return s;
}

// n streams from P.from to P.to at the rate of h's operator: one launch of the copy path
static int launch_copy(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const capy_hasher* h, uint64_t n, SpongeCopy P) {
  if (n == 0) return CAPY_OK;
  SpongeJob J = hasher_operator(h);
  J.n = n;
  P.on = 1;
  return launch_chain_jobs(ctx, dc, st, J, J, false, 1, nullptr, nullptr, nullptr, &P);
}

// a device copy of v (kept alive by p) on st; v must outlive the copy
static int upload(capy_ctx* ctx, cudaStream_t st, DevPtr<uint64_t>& p, const std::vector<uint64_t>& v) {
  if (v.empty()) return CAPY_OK;
  if (dev_alloc(p, v.size() * 8) != cudaSuccess) {
    cudaGetLastError();
    return CAPY_ERR_OOM;
  }
  CAPY_CUDA(ctx, cudaMemcpyAsync(p.get(), v.data(), v.size() * 8, cudaMemcpyHostToDevice, st));
  return CAPY_OK;
}

// Item j of f starts as a copy of item src[j] of h (same ctx).  A destination device b copies the sources it holds itself
// in one launch with both maps.  Sources on another device a are gathered there into compact records, moved to b with one
// peer copy and scattered.  Blocking: every phase ends in stream synchronisations before the next one reads its results.
static int fork_items(capy_ctx* ctx, const capy_hasher* h, const uint64_t* src, capy_hasher* f) {
  const size_t nd = ctx->devs.size();
  const uint64_t rec = blob_record(h->rate);
  // s_loc[a][b] / d_loc[a][b]: the sources on device a of the destinations on device b, as indices on a and on b
  std::vector<std::vector<std::vector<uint64_t>>> s_loc(nd, std::vector<std::vector<uint64_t>>(nd)), d_loc = s_loc;
  for (size_t b = 0; b < nd; b++)
    for (uint64_t j = f->first[b]; j < f->first[b + 1]; j++) {
      const size_t a = (size_t)(std::upper_bound(h->first.begin(), h->first.end(), src[j]) - h->first.begin()) - 1;
      s_loc[a][b].push_back(src[j] - h->first[a]);
      d_loc[a][b].push_back(j - f->first[b]);
    }
  std::vector<std::vector<DevPtr<uint8_t>>> moved(nd);  // [a][b]: records gathered on a for b
  std::vector<std::vector<DevPtr<uint64_t>>> maps(nd);
  for (size_t a = 0; a < nd; a++) {
    moved[a].resize(nd);
    maps[a].resize(2 * nd);
  }
  for (size_t a = 0; a < nd; a++) {  // gather
    DeviceCtx& dc = ctx->devs[a];
    std::lock_guard<std::mutex> lk(*dc.mu);
    DeviceGuard g(dc.dev);
    const cudaStream_t st = dc.streams[0];
    for (size_t b = 0; b < nd; b++) {
      const uint64_t cnt = s_loc[a][b].size();
      if (b == a || cnt == 0) continue;
      if (dev_alloc(moved[a][b], cnt * rec) != cudaSuccess) {
        cudaGetLastError();
        return CAPY_ERR_OOM;
      }
      int rc = upload(ctx, st, maps[a][b], s_loc[a][b]);
      SpongeCopy P{};
      P.src = maps[a][b].get();
      P.from = hasher_side(h, (int)a, 0);
      P.to = record_side(moved[a][b].get());
      if (!rc) rc = launch_copy(ctx, dc, st, h, cnt, P);
      if (rc) return rc;
    }
    CAPY_CUDA(ctx, cudaStreamSynchronize(st));
  }
  for (size_t b = 0; b < nd; b++) {  // move and scatter, or copy in place
    DeviceCtx& dc = ctx->devs[b];
    std::lock_guard<std::mutex> lk(*dc.mu);
    DeviceGuard g(dc.dev);
    const cudaStream_t st = dc.streams[0];
    std::vector<DevPtr<uint8_t>> here(nd);
    for (size_t a = 0; a < nd; a++) {
      const uint64_t cnt = s_loc[a][b].size();
      if (cnt == 0) continue;
      SpongeCopy P{};
      P.to = hasher_side(f, (int)b, 0);
      int rc = CAPY_OK;
      if (cnt < hasher_items(f, (int)b)) rc = upload(ctx, st, maps[b][nd + a], d_loc[a][b]);  // else the identity
      P.dst = maps[b][nd + a].get();
      if (a == b) {
        if (!rc) rc = upload(ctx, st, maps[b][b], s_loc[b][b]);
        P.src = maps[b][b].get();
        P.from = hasher_side(h, (int)b, 0);
      } else {
        if (!rc && dev_alloc(here[a], cnt * rec) != cudaSuccess) {
          cudaGetLastError();
          rc = CAPY_ERR_OOM;
        }
        if (!rc) {
          const cudaError_t e = cudaMemcpyPeerAsync(here[a].get(), dc.dev, moved[a][b].get(), ctx->devs[a].dev, cnt * rec, st);
          if (e != cudaSuccess) rc = cuda_fail(ctx, e, "cudaMemcpyPeerAsync");
        }
        P.from = record_side(here[a].get());
      }
      if (!rc) rc = launch_copy(ctx, dc, st, h, cnt, P);
      if (rc) {
        cudaStreamSynchronize(st);  // (the buffers of this device go back after the work that reads them)
        return rc;
      }
    }
    CAPY_CUDA(ctx, cudaStreamSynchronize(st));
  }
  return CAPY_OK;
}

}  // namespace capy

using namespace capy;

extern "C" {

// =================================================================================================
// diagnostics
// =================================================================================================
int capy_plan_tiers(const uint32_t* items_longer_than, uint32_t n_bins, uint64_t n, uint32_t max_blocks, uint64_t total_blocks,
                    int sm_count, uint64_t* warp_items, uint64_t* pair_items) {
  uint64_t w[3];
  int rc = capy_plan_tiers3(items_longer_than, n_bins, n, max_blocks, total_blocks, sm_count, w, pair_items);
  if (rc == CAPY_OK && warp_items) *warp_items = w[0] + w[1] + w[2];
  return warp_items ? rc : CAPY_ERR_BAD_ARG;
}

int capy_plan_tiers3(const uint32_t* items_longer_than, uint32_t n_bins, uint64_t n, uint32_t max_blocks, uint64_t total_blocks,
                     int sm_count, uint64_t* warp_items_by_sharing, uint64_t* pair_items) {
  if (!items_longer_than || !n_bins || !warp_items_by_sharing || !pair_items || sm_count < 2) return CAPY_ERR_BAD_ARG;
  std::vector<uint32_t> cum(items_longer_than, items_longer_than + n_bins);
  plan_tiers(cum, n, max_blocks, (double)total_blocks, sm_count, warp_items_by_sharing, pair_items);
  return CAPY_OK;
}

int capy_chain_cut(int sm_count, uint64_t n, uint64_t absorb_blocks, uint64_t squeeze_extra, uint64_t* cut_after_blocks) {
  if (!cut_after_blocks) return CAPY_ERR_BAD_ARG;
  *cut_after_blocks = 0;
  return chain_cut(sm_count, n, absorb_blocks, squeeze_extra, cut_after_blocks) ? 1 : 0;
}

int capy_lpt_shares(const uint64_t* off, uint64_t n, uint32_t parts, uint32_t unit_bytes, uint64_t per_item_cost,
                    uint32_t* owner) {
  if (!off || !owner || parts == 0 || unit_bytes == 0) return CAPY_ERR_BAD_ARG;
  auto shares = lpt_shares(off, n, parts, unit_bytes, per_item_cost);
  for (size_t d = 0; d < shares.size(); d++)
    for (const Run& r : shares[d].runs)
      for (uint64_t i = r.i0; i < r.i1; i++) owner[i] = (uint32_t)d;
  return CAPY_OK;
}

// =================================================================================================
// SHA3-d
// =================================================================================================
int capy_sha3_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_data,
                        const uint64_t* d_off, uint64_t n, uint8_t* d_digests, uint32_t flags) {
  if (n && (!d_data || !d_off || !d_digests)) return CAPY_ERR_BAD_ARG;
  CAPY_DEV_PROLOGUE
  return launch_sha3(ctx, dc, st, d_bits, d_data, d_off, 0, 0, n, d_digests, flags);
}

int capy_sha3_batch_fixed_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_data,
                              uint64_t msg_len, uint64_t stride, uint64_t n, uint8_t* d_digests, uint32_t) {
  if ((n && (!d_data || !d_digests)) || stride < msg_len) return CAPY_ERR_BAD_ARG;
  CAPY_DEV_PROLOGUE
  return launch_sha3(ctx, dc, st, d_bits, d_data, nullptr, msg_len, stride, n, d_digests, 0, /*tail_readable=*/false);
}

int capy_sha3_batch(capy_ctx* ctx, int d_bits, const uint8_t* data, const uint64_t* off, uint64_t n, uint8_t* digests,
                    uint32_t flags) {
  if (!ctx || (n && (!data || !off || !digests))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  const size_t ob = (size_t)d_bits / 8;
  if (ctx->devs.size() > 1) {
    // several devices: the outliers of the batch (long chains) are dealt out longest first, the rest follows in
    // contiguous ranges (lpt_shares).  When nothing had to be dealt out every share is one run and the plain path
    // below does the same thing with pipelined chunks.
    auto shares = lpt_shares(off, n, ctx->devs.size(), sha3_rate(d_bits), 2);
    bool scattered = false;
    for (const DeviceShare& s : shares) scattered |= s.runs.size() > 1;
    if (scattered) {
      std::vector<Range> slots;
      for (size_t k = 0; k < shares.size(); k++) slots.push_back({k, k + 1});  // for_each_device: one closure per device
      return for_each_device(ctx, slots, [&](DeviceCtx& dc, Range slot, int*) -> int {
        const DeviceShare& sh = shares[slot.i0];
        if (sh.items == 0) return CAPY_OK;
        cudaStream_t st = dc.streams[0];
        uint8_t* d_data = (uint8_t*)scratch_get(dc, st, kHost0, (size_t)sh.bytes + 16);
        uint64_t* d_off = (uint64_t*)scratch_get(dc, st, kHost1, (size_t)(sh.items + 1) * 8);
        uint8_t* d_out = (uint8_t*)scratch_get(dc, st, kHost2, (size_t)sh.items * ob);
        if (!d_data || !d_off || !d_out) return CAPY_ERR_OOM;
        std::vector<uint64_t> loc(sh.items + 1);  // offsets of this device's items in its own packed buffer
        uint64_t at = 0, j = 0;
        for (const Run& r : sh.runs) {  // one copy per run of consecutive messages
          const uint64_t b0 = off[r.i0], b1 = off[r.i1];
          if (b1 > b0) {
            const int rc = copy_in(ctx, dc, st, kHost0, d_data + at, data + b0, (size_t)(b1 - b0));
            if (rc) return rc;
          }
          for (uint64_t i = r.i0; i < r.i1; i++) loc[j++] = at + (off[i] - b0);
          at += b1 - b0;
        }
        loc[j] = at;
        CAPY_CUDA(ctx, cudaMemcpyAsync(d_off, loc.data(), (size_t)(sh.items + 1) * 8, cudaMemcpyHostToDevice, st));
        host_off_register(dc, d_off, loc.data(), sh.items + 1);
        int rc = launch_sha3(ctx, dc, st, d_bits, d_data, d_off, 0, 0, sh.items, d_out, flags);
        if (rc) return rc;
        j = 0;
        for (const Run& r : sh.runs) {  // the digests of a run are consecutive on both sides
          rc = copy_out(ctx, dc, st, kHost2, digests + r.i0 * ob, d_out + j * ob, (size_t)(r.i1 - r.i0) * ob);
          if (rc) return rc;
          j += r.i1 - r.i0;
        }
        CAPY_CUDA(ctx, cudaStreamSynchronize(st));  // (`loc` stays alive until here)
        return CAPY_OK;
      });
    }
  }
  auto shards = split_items(off, 0, 0, n, ctx->devs.size(), 200);
  // long messages: few big chunks, so that the longest-first schedule sees enough work beside them
  auto chunks = [&](Range sh) { return split_items(off, 0, sh.i0, sh.i1, ragged_chunk_count(off, sh.i0, sh.i1, 0), 200); };
  return run_host_call(ctx, shards, chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(data, off);
    uint8_t* d_out = io.out(digests, ob);
    if (io.rc()) return io.rc();
    return launch_sha3(ctx, dc, st, d_bits, sp.d_base, sp.d_off, 0, 0, io.n(), d_out, flags);
  });
}

int capy_sha3_batch_fixed(capy_ctx* ctx, int d_bits, const uint8_t* data, uint64_t msg_len, uint64_t stride, uint64_t n,
                          uint8_t* digests, uint32_t) {
  if (!ctx || (n && (!data || !digests)) || stride < msg_len) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  const size_t ob = (size_t)d_bits / 8;
  // the uniform kernel wants 8-byte aligned rows; the copy lands on a 256-byte aligned buffer, so
  // only the stride matters
  auto shards = split_items(nullptr, stride, 0, n, ctx->devs.size(), 0);
  auto chunks = [&](Range sh) {
    return split_items(nullptr, stride, sh.i0, sh.i1, chunk_count((sh.i1 - sh.i0) * stride, sh.i1 - sh.i0), 0);
  };
  return run_host_call(ctx, shards, chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    // the last row may be shorter than the stride in the caller's buffer
    const uint8_t* d_in = io.in(data, stride, (size_t)((io.n() - 1) * stride + msg_len));
    uint8_t* d_out = io.out(digests, ob);
    if (io.rc()) return io.rc();
    return launch_sha3(ctx, dc, st, d_bits, d_in, nullptr, msg_len, stride, io.n(), d_out);
  });
}

// =================================================================================================
// cSHAKE
// =================================================================================================
int capy_cshake_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_data,
                          const uint64_t* d_off, uint64_t n, const uint8_t* fn_name, uint32_t fn_len,
                          const uint8_t* custom, uint32_t custom_len, uint64_t out_bits, uint8_t* d_out) {
  if ((n && (!d_data || !d_off || !d_out)) || (fn_len && !fn_name) || (custom_len && !custom)) return CAPY_ERR_BAD_ARG;
  CAPY_DEV_PROLOGUE
  return launch_cshake(ctx, dc, st, d_bits, d_data, d_off, n, fn_name, fn_len, custom, custom_len, out_bits, d_out);
}

int capy_cshake_batch(capy_ctx* ctx, int d_bits, const uint8_t* data, const uint64_t* off, uint64_t n,
                      const uint8_t* fn_name, uint32_t fn_len, const uint8_t* custom, uint32_t custom_len,
                      uint64_t out_bits, uint8_t* out) {
  if (!ctx || (n && (!data || !off || !out)) || (fn_len && !fn_name) || (custom_len && !custom)) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  const size_t ob = (size_t)(out_bits / 8);
  if (n == 0 || ob == 0) return CAPY_OK;
  auto shards = split_items(off, 0, 0, n, ctx->devs.size(), 200 + ob);
  auto chunks = [&](Range sh) {
    return split_items(off, 0, sh.i0, sh.i1, ragged_chunk_count(off, sh.i0, sh.i1, (sh.i1 - sh.i0) * ob), 200 + ob);
  };
  return run_host_call(ctx, shards, chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(data, off);
    uint8_t* d_out = io.out(out, ob);
    if (io.rc()) return io.rc();
    return launch_cshake(ctx, dc, st, d_bits, sp.d_base, sp.d_off, io.n(), fn_name, fn_len, custom, custom_len, out_bits,
                         d_out);
  });
}

// =================================================================================================
// KMACXOF
// =================================================================================================
int capy_kmac_xof_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_keys,
                            const uint64_t* d_key_off, const uint8_t* d_data, const uint64_t* d_off, uint64_t n,
                            const uint8_t* custom, uint32_t custom_len, uint64_t out_bits, const uint64_t* d_out_off,
                            uint8_t* d_out) {
  if ((n && (!d_keys || !d_key_off || !d_data || !d_off || !d_out)) || (custom_len && !custom)) return CAPY_ERR_BAD_ARG;
  CAPY_DEV_PROLOGUE
  KmacPass a(d_bits, {reinterpret_cast<const char*>(custom), custom_len}, n);
  a.job.keys = d_keys;
  a.job.key_off = d_key_off;
  a.job.data = d_data;
  a.job.off = d_off;
  a.job.out_bytes = a.job.out_stride = out_bits / 8;
  a.job.out_off = d_out_off;
  a.job.out = d_out;
  return launch_kmac_xof(ctx, dc, st, a);
}

int capy_kmac_xof_batch_fixed_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_keys,
                                  uint64_t key_len, uint64_t key_stride, const uint8_t* d_data, uint64_t msg_len,
                                  uint64_t msg_stride, uint64_t n, const uint8_t* custom, uint32_t custom_len,
                                  uint64_t out_bits, uint8_t* d_out) {
  if ((n && (!d_keys || !d_out)) || (n && msg_len && !d_data) || (custom_len && !custom) || key_stride < key_len ||
      msg_stride < msg_len)
    return CAPY_ERR_BAD_ARG;
  CAPY_DEV_PROLOGUE
  KmacPass a(d_bits, {reinterpret_cast<const char*>(custom), custom_len}, n);
  a.job.keys = d_keys;
  a.job.key_len = (uint32_t)key_len;
  a.job.key_stride = key_stride;
  a.job.data = d_data;
  a.job.msg_len = msg_len;
  a.job.msg_stride = msg_stride;
  a.job.out_bytes = a.job.out_stride = out_bits / 8;
  a.job.out = d_out;
  return launch_kmac_xof(ctx, dc, st, a);
}

int capy_kmac_xof_batch(capy_ctx* ctx, int d_bits, const uint8_t* keys, const uint64_t* key_off, const uint8_t* data,
                        const uint64_t* off, uint64_t n, const uint8_t* custom, uint32_t custom_len, uint64_t out_bits,
                        const uint64_t* out_off, uint8_t* out) {
  if (!ctx || (n && (!keys || !key_off || !data || !off || !out)) || (custom_len && !custom)) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  const size_t ob = (size_t)(out_bits / 8);
  if (n == 0 || (!out_off && ob == 0)) return CAPY_OK;
  auto out_begin = [&](uint64_t i) -> uint64_t { return out_off ? out_off[i] : i * ob; };
  auto shards = split_items(off, 0, 0, n, ctx->devs.size(), 400 + ob);
  auto chunks = [&](Range sh) {
    return split_items(off, 0, sh.i0, sh.i1, ragged_chunk_count(off, sh.i0, sh.i1, out_begin(sh.i1) - out_begin(sh.i0)),
                       400 + ob);
  };
  return run_host_call(ctx, shards, chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sx = io.in_packed(data, off), sk = io.in_packed(keys, key_off);
    KmacPass a(d_bits, {reinterpret_cast<const char*>(custom), custom_len}, io.n());
    a.job.keys = sk.d_base;
    a.job.key_off = sk.d_off;
    a.job.data = sx.d_base;
    a.job.off = sx.d_off;
    a.job.out_bytes = a.job.out_stride = ob;
    if (out_off) {
      a.job.out_off = (const uint64_t*)io.in(out_off, 8, (size_t)(io.n() + 1) * 8);
      a.job.out = io.out_packed(out, out_off);
    } else {
      a.job.out = io.out(out, ob);
    }
    if (io.rc()) return io.rc();
    return launch_kmac_xof(ctx, dc, st, a);
  });
}

// =================================================================================================
// FIPS 202 SHAKE (no reference counterpart)
// =================================================================================================
int capy_fips_shake_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int shake_bits, const uint8_t* d_data,
                              const uint64_t* d_off, uint64_t n, uint64_t out_bytes, uint8_t* d_out) {
  if (!dev_index_ok(ctx, dev_index) || (n && (!d_data || !d_off || !d_out)) || (shake_bits != 128 && shake_bits != 256))
    return CAPY_ERR_BAD_ARG;
  if (n == 0 || out_bytes == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  SpongeJob J = shake_job(shake_bits);
  J.data = d_data;
  J.off = d_off;
  J.out = d_out;
  J.out_stride = J.out_bytes = out_bytes;
  J.n = n;
  LaunchPlan plan;  // longest first, tiers for chain-bound batches, chains of a uniform batch cut in two: as for cSHAKE
  int rc = plan_ragged(ctx, dc, st, d_off, n, J.rate, &plan);
  if (rc) return rc;
  return run_sponge(ctx, dc, st, J, plan);
}

// =================================================================================================
// resumable SHA3-d / KMACXOF streams
// =================================================================================================
int capy_sha3_hasher_new(capy_ctx* ctx, int d_bits, uint64_t n, capy_hasher** out) {
  if (!out) return CAPY_ERR_BAD_ARG;
  *out = nullptr;
  if (!ctx) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  return hasher_create(ctx, d_bits, kSha3Stream, n, out);
}

int capy_kmac_xof_hasher_new(capy_ctx* ctx, int d_bits, const uint8_t* keys, const uint64_t* key_off, uint64_t n,
                             const uint8_t* custom, uint32_t custom_len, capy_hasher** out) {
  if (!out) return CAPY_ERR_BAD_ARG;
  *out = nullptr;
  if (!ctx || (n && (!keys || !key_off)) || (custom_len && !custom)) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (d_bits == 224) return CAPY_ERR_BAD_ARG;  // the 172-byte rate is read as 168 (Q7): see the header
  capy_hasher* h = nullptr;
  int rc = hasher_create(ctx, d_bits, kKmacStream, n, &h);
  if (rc || n == 0) {
    *out = h;
    return rc;
  }
  // P | KB: the cached prefix state, then the key block of every item (one chunk per device: the states are stored at
  // [k * n + i])
  rc = run_host_call(ctx, hasher_shards(h), one_chunk, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    if (io.n() == 0) return CAPY_OK;  // (a device without items)
    const StagedPacked sk = io.in_packed(keys, key_off);
    if (io.rc()) return io.rc();
    KmacPass a(d_bits, {reinterpret_cast<const char*>(custom), custom_len}, io.n());
    a.job.keys = sk.d_base;
    a.job.key_off = sk.d_off;
    return launch_kmac_state(ctx, dc, st, a, false, h->d_state[dc.index]);
  });
  if (rc) {
    capy_hasher_free(h);
    return rc;
  }
  *out = h;
  return CAPY_OK;
}

int capy_hasher_device_range(const capy_hasher* h, int dev_index, uint64_t* i0, uint64_t* i1) {
  if (!h || !i0 || !i1 || dev_index < 0 || dev_index >= (int)h->dev.size()) return CAPY_ERR_BAD_ARG;
  *i0 = h->first[dev_index];
  *i1 = h->first[dev_index + 1];
  return CAPY_OK;
}

int capy_hasher_update(capy_ctx* ctx, capy_hasher* h, const uint8_t* data, const uint64_t* off) {
  if (hasher_check(ctx, h) || h->kind == kEncryptStream || hasher_any_finished(h) || (h->n && (!data || !off)))
    return CAPY_ERR_BAD_ARG;
  if (h->kind == kDecryptStream && !hasher_in_pass(h, kDecryptStream, 1)) return CAPY_ERR_BAD_ARG;  // pass 2: decrypt_update
  if (h->n == 0) return CAPY_OK;
  auto chunks = [&](Range sh) {
    return split_items(off, 0, sh.i0, sh.i1, chunk_count(off[sh.i1] - off[sh.i0], sh.i1 - sh.i0), 200);
  };
  return run_host_call(ctx, hasher_shards(h), chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(data, off);
    if (io.rc()) return io.rc();
    return hasher_piece_items(ctx, dc, st, h, io.i0() - h->first[dc.index], io.n(), sp.d_base, sp.d_off);
  });
}

int capy_hasher_update_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, const uint8_t* d_data,
                           const uint64_t* d_off) {
  if (hasher_check(ctx, h) || h->kind == kEncryptStream || !dev_index_ok(ctx, dev_index) || h->finished[dev_index])
    return CAPY_ERR_BAD_ARG;
  if (h->kind == kDecryptStream && h->pass[dev_index] != 1) return CAPY_ERR_BAD_ARG;
  const uint64_t m = hasher_items(h, dev_index);
  if (m && (!d_data || !d_off)) return CAPY_ERR_BAD_ARG;
  if (m == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  return hasher_piece_items(ctx, dc, st, h, 0, m, d_data, d_off);
}

int capy_hasher_final(capy_ctx* ctx, capy_hasher* h, uint64_t out_bits, const uint64_t* out_off, uint8_t* out) {
  if (hasher_check(ctx, h) || hasher_any_finished(h) || (h->n && !out)) return CAPY_ERR_BAD_ARG;
  if (!hasher_final_fits(h, out_bits, out_off)) return CAPY_ERR_BAD_ARG;
  for (char& f : h->finished) f = 1;
  const size_t ob = (size_t)(out_bits / 8);
  if (h->n == 0 || (!out_off && ob == 0)) return CAPY_OK;
  auto out_begin = [&](uint64_t i) -> uint64_t { return out_off ? out_off[i] : i * ob; };
  auto chunks = [&](Range sh) {
    return split_items(out_off, ob, sh.i0, sh.i1, chunk_count(out_begin(sh.i1) - out_begin(sh.i0), sh.i1 - sh.i0), 0);
  };
  return run_host_call(ctx, hasher_shards(h), chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const uint64_t* d_out_off = nullptr;
    uint8_t* d_out;
    if (out_off) {
      d_out_off = (const uint64_t*)io.in(out_off, 8, (size_t)(io.n() + 1) * 8);
      d_out = io.out_packed(out, out_off);
    } else {
      d_out = io.out(out, ob);
    }
    if (io.rc()) return io.rc();
    return hasher_final_items(ctx, dc, st, h, io.i0() - h->first[dc.index], io.n(), ob, d_out_off, d_out);
  });
}

int capy_hasher_final_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint64_t out_bits,
                          const uint64_t* d_out_off, uint8_t* d_out) {
  if (hasher_check(ctx, h) || !dev_index_ok(ctx, dev_index) || h->finished[dev_index]) return CAPY_ERR_BAD_ARG;
  if (!hasher_final_fits(h, out_bits, d_out_off)) return CAPY_ERR_BAD_ARG;
  const uint64_t m = hasher_items(h, dev_index);
  if (m && !d_out) return CAPY_ERR_BAD_ARG;
  h->finished[dev_index] = 1;
  if (m == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  return hasher_final_items(ctx, dc, st, h, 0, m, out_bits / 8, d_out_off, d_out);
}

// ---- encryption and verification streams (created in ae_api.cu and ed448_api.cu) -------------------------------------
int capy_hasher_encrypt_update(capy_ctx* ctx, capy_hasher* h, const uint8_t* data, const uint64_t* off, uint8_t* ct) {
  if (hasher_check(ctx, h) || h->kind != kEncryptStream || hasher_any_finished(h) || (h->n && (!data || !off || !ct)))
    return CAPY_ERR_BAD_ARG;
  if (h->n == 0) return CAPY_OK;
  auto chunks = [&](Range sh) {
    return split_items(off, 0, sh.i0, sh.i1, chunk_count(off[sh.i1] - off[sh.i0], sh.i1 - sh.i0), 400);
  };
  return run_host_call(ctx, hasher_shards(h), chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(data, off);
    uint8_t* d_ct = io.out_packed(ct, off);
    if (io.rc()) return io.rc();
    return hasher_encrypt_items(ctx, dc, st, h, io.i0() - h->first[dc.index], io.n(), sp.d_base, sp.d_off, d_ct);
  });
}

int capy_hasher_encrypt_update_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, const uint8_t* d_data,
                                   const uint64_t* d_off, uint8_t* d_ct) {
  if (hasher_check(ctx, h) || h->kind != kEncryptStream || !dev_index_ok(ctx, dev_index) || h->finished[dev_index])
    return CAPY_ERR_BAD_ARG;
  const uint64_t m = hasher_items(h, dev_index);
  if (m && (!d_data || !d_off || !d_ct)) return CAPY_ERR_BAD_ARG;
  if (m == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  return hasher_encrypt_items(ctx, dc, st, h, 0, m, d_data, d_off, d_ct);
}

int capy_hasher_verify_final(capy_ctx* ctx, capy_hasher* h, uint8_t* ok) {
  if (hasher_check(ctx, h) || h->kind != kVerifyStream || hasher_any_finished(h) || (h->n && !ok)) return CAPY_ERR_BAD_ARG;
  for (char& f : h->finished) f = 1;
  if (h->n == 0) return CAPY_OK;
  return run_host_call(ctx, hasher_shards(h), one_chunk, true, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    uint8_t* d_ok = io.out(ok, 1);
    if (io.rc()) return io.rc();
    return hasher_verify_items(ctx, dc, st, h, io.i0() - h->first[dc.index], io.n(), d_ok, io.d_flag());
  });
}

int capy_hasher_verify_final_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint8_t* d_ok, int* d_bad_flag) {
  if (hasher_check(ctx, h) || h->kind != kVerifyStream || !dev_index_ok(ctx, dev_index) || h->finished[dev_index])
    return CAPY_ERR_BAD_ARG;
  const uint64_t m = hasher_items(h, dev_index);
  if (m && !d_ok) return CAPY_ERR_BAD_ARG;
  h->finished[dev_index] = 1;
  if (m == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  return hasher_verify_items(ctx, dc, st, h, 0, m, d_ok, d_bad_flag);
}

// ---- sign and decryption streams: two passes (created in ed448_api.cu and ae_api.cu) ----------------------------------
// The pass moves to 2 before the device work of next_pass runs, as `finished` does before a final: a next_pass that fails
// (an OOM, a CUDA error) leaves its streams with half-updated states, and the only call left that is of use is
// capy_hasher_free.
int capy_hasher_next_pass(capy_ctx* ctx, capy_hasher* h, uint8_t* ok) {
  if (hasher_check(ctx, h)) return CAPY_ERR_BAD_ARG;
  const bool sign = hasher_in_pass(h, kSignStream, 1), dec = hasher_in_pass(h, kDecryptStream, 1);
  if ((!sign && !dec) || (sign && ok)) return CAPY_ERR_BAD_ARG;
  for (char& p : h->pass) p = 2;
  if (h->n == 0) return CAPY_OK;
  return run_host_call(ctx, hasher_shards(h), one_chunk, dec && h->tag_bits == 448,
                       [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    if (io.n() == 0) return CAPY_OK;  // (a device without items)
    uint8_t* d_ok = ok ? io.out(ok, 1) : nullptr;
    if (io.rc()) return io.rc();
    return sign ? sign_stream_next(ctx, dc, st, h) : decrypt_stream_check(ctx, dc, st, h, false, d_ok, io.d_flag());
  });
}

int capy_hasher_next_pass_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint8_t* d_ok, int* d_bad_flag) {
  if (hasher_check(ctx, h) || !dev_index_ok(ctx, dev_index)) return CAPY_ERR_BAD_ARG;
  const bool sign = hasher_dev_in_pass(h, dev_index, kSignStream, 1), dec = hasher_dev_in_pass(h, dev_index, kDecryptStream, 1);
  if ((!sign && !dec) || (sign && d_ok)) return CAPY_ERR_BAD_ARG;
  h->pass[dev_index] = 2;
  if (hasher_items(h, dev_index) == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  return sign ? sign_stream_next(ctx, dc, st, h) : decrypt_stream_check(ctx, dc, st, h, false, d_ok, d_bad_flag);
}

int capy_hasher_decrypt_update(capy_ctx* ctx, capy_hasher* h, const uint8_t* ct, const uint64_t* off, uint8_t* out) {
  if (hasher_check(ctx, h) || !hasher_in_pass(h, kDecryptStream, 2) || (h->n && (!ct || !off || !out))) return CAPY_ERR_BAD_ARG;
  if (h->n == 0) return CAPY_OK;
  auto chunks = [&](Range sh) {
    return split_items(off, 0, sh.i0, sh.i1, chunk_count(off[sh.i1] - off[sh.i0], sh.i1 - sh.i0), 400);
  };
  return run_host_call(ctx, hasher_shards(h), chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(ct, off);
    uint8_t* d_out = io.out_packed(out, off);
    if (io.rc()) return io.rc();
    return hasher_dual_items(ctx, dc, st, h, io.i0() - h->first[dc.index], io.n(), sp.d_base, sp.d_off, d_out);
  });
}

int capy_hasher_decrypt_update_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, const uint8_t* d_ct,
                                   const uint64_t* d_off, uint8_t* d_out) {
  if (hasher_check(ctx, h) || !dev_index_ok(ctx, dev_index) || !hasher_dev_in_pass(h, dev_index, kDecryptStream, 2))
    return CAPY_ERR_BAD_ARG;
  const uint64_t m = hasher_items(h, dev_index);
  if (m && (!d_ct || !d_off || !d_out)) return CAPY_ERR_BAD_ARG;
  if (m == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  return hasher_dual_items(ctx, dc, st, h, 0, m, d_ct, d_off, d_out);
}

int capy_hasher_decrypt_final(capy_ctx* ctx, capy_hasher* h, uint8_t* ok) {
  if (hasher_check(ctx, h) || !hasher_in_pass(h, kDecryptStream, 2) || (h->n && !ok)) return CAPY_ERR_BAD_ARG;
  for (char& f : h->finished) f = 1;
  if (h->n == 0) return CAPY_OK;
  return run_host_call(ctx, hasher_shards(h), one_chunk, h->tag_bits == 448,
                       [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    if (io.n() == 0) return CAPY_OK;
    uint8_t* d_ok = io.out(ok, 1);
    if (io.rc()) return io.rc();
    return decrypt_stream_check(ctx, dc, st, h, true, d_ok, io.d_flag());
  });
}

int capy_hasher_decrypt_final_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint8_t* d_ok, int* d_bad_flag) {
  if (hasher_check(ctx, h) || !dev_index_ok(ctx, dev_index) || !hasher_dev_in_pass(h, dev_index, kDecryptStream, 2))
    return CAPY_ERR_BAD_ARG;
  const uint64_t m = hasher_items(h, dev_index);
  if (m && !d_ok) return CAPY_ERR_BAD_ARG;
  h->finished[dev_index] = 1;
  if (m == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  return decrypt_stream_check(ctx, dc, st, h, true, d_ok, d_bad_flag);
}

int capy_hasher_sign_final(capy_ctx* ctx, capy_hasher* h, uint8_t* h56, uint8_t* z_be56, uint8_t* ok) {
  if (hasher_check(ctx, h) || !hasher_in_pass(h, kSignStream, 2) || (h->n && (!h56 || !z_be56 || !ok)))
    return CAPY_ERR_BAD_ARG;
  for (char& f : h->finished) f = 1;
  if (h->n == 0) return CAPY_OK;
  return run_host_call(ctx, hasher_shards(h), one_chunk, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    if (io.n() == 0) return CAPY_OK;
    uint8_t* d_h = io.out(h56, 56);
    uint8_t* d_z = io.out(z_be56, 56);
    uint8_t* d_ok = io.out(ok, 1);
    if (io.rc()) return io.rc();
    return sign_stream_final(ctx, dc, st, h, d_h, d_z, d_ok);
  });
}

int capy_hasher_sign_final_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint8_t* d_h56, uint8_t* d_z_be56,
                               uint8_t* d_ok) {
  if (hasher_check(ctx, h) || !dev_index_ok(ctx, dev_index) || !hasher_dev_in_pass(h, dev_index, kSignStream, 2))
    return CAPY_ERR_BAD_ARG;
  const uint64_t m = hasher_items(h, dev_index);
  if (m && (!d_h56 || !d_z_be56 || !d_ok)) return CAPY_ERR_BAD_ARG;
  h->finished[dev_index] = 1;
  if (m == 0) return CAPY_OK;
  CAPY_DEV_PROLOGUE
  return sign_stream_final(ctx, dc, st, h, d_h56, d_z_be56, d_ok);
}

// ---- checkpoints and forks of SHA3-d / KMACXOF streams --------------------------------------------------------------
int capy_hasher_export_size(const capy_hasher* h, uint64_t* bytes) {
  if (!h || !bytes || !hasher_portable(h)) return CAPY_ERR_BAD_ARG;
  *bytes = kBlobHeader + h->n * blob_record(h->rate);
  return CAPY_OK;
}

int capy_hasher_export(capy_ctx* ctx, const capy_hasher* h, uint8_t* blob, uint64_t blob_len) {
  if (hasher_check(ctx, h) || !hasher_portable(h) || !blob) return CAPY_ERR_BAD_ARG;
  const uint64_t rec = blob_record(h->rate);
  if (blob_len < kBlobHeader + h->n * rec) return CAPY_ERR_BAD_ARG;
  uint8_t hdr[kBlobHeader] = {};
  memcpy(hdr, kBlobMagic, 8);
  put_le(hdr + 8, kBlobVersion, 4);
  put_le(hdr + 12, h->kind == kKmacStream ? 1 : 0, 4);
  put_le(hdr + 16, (uint64_t)h->d_bits, 4);
  put_le(hdr + 20, h->rate, 4);
  put_le(hdr + 24, rec, 4);
  put_le(hdr + 32, h->n, 8);
  memcpy(blob, hdr, kBlobHeader);
  if (h->n == 0) return CAPY_OK;
  auto chunks = [&](Range sh) {
    return split_items(nullptr, rec, sh.i0, sh.i1, chunk_count((sh.i1 - sh.i0) * rec, sh.i1 - sh.i0), 0);
  };
  return run_host_call(ctx, hasher_shards(h), chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    uint8_t* d_rec = io.out(blob + kBlobHeader, rec);
    if (io.rc()) return io.rc();
    SpongeCopy P{};
    P.from = hasher_side(h, dc.index, io.i0() - h->first[dc.index]);
    P.to = record_side(d_rec);
    return launch_copy(ctx, dc, st, h, io.n(), P);
  });
}

int capy_hasher_blob_info(const uint8_t* blob, uint64_t blob_len, int* kind, int* d_bits, uint64_t* n) {
  BlobHeader b;
  const int rc = blob_parse(blob, blob_len, &b);
  if (rc) return rc;
  if (kind) *kind = b.kind == kKmacStream ? 1 : 0;
  if (d_bits) *d_bits = b.d_bits;
  if (n) *n = b.n;
  return CAPY_OK;
}

int capy_hasher_import(capy_ctx* ctx, const uint8_t* blob, uint64_t blob_len, capy_hasher** out) {
  if (!out) return CAPY_ERR_BAD_ARG;
  *out = nullptr;
  BlobHeader b;
  if (!ctx || blob_parse(blob, blob_len, &b)) return CAPY_ERR_BAD_ARG;
  capy_hasher* h = nullptr;
  int rc = hasher_create(ctx, b.d_bits, b.kind, b.n, &h);
  if (rc) return rc;
  const uint64_t rec = blob_record(b.rate);
  auto chunks = [&](Range sh) {
    return split_items(nullptr, rec, sh.i0, sh.i1, chunk_count((sh.i1 - sh.i0) * rec, sh.i1 - sh.i0), 0);
  };
  // a record with a non-zero carry tail raises the chunk's flag, which run_host_call reports as a bad point
  rc = run_host_call(ctx, hasher_shards(h), chunks, true, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const uint8_t* d_rec = io.in(blob + kBlobHeader, rec);
    if (io.rc()) return io.rc();
    SpongeCopy P{};
    P.from = record_side(const_cast<uint8_t*>(d_rec));
    P.to = hasher_side(h, dc.index, io.i0() - h->first[dc.index]);
    P.bad_tail = io.d_flag();
    return launch_copy(ctx, dc, st, h, io.n(), P);
  });
  if (rc) {
    capy_hasher_free(h);
    return rc == CAPY_ERR_BAD_POINT ? CAPY_ERR_BAD_ARG : rc;
  }
  *out = h;
  return CAPY_OK;
}

int capy_hasher_fork(capy_ctx* ctx, const capy_hasher* h, const uint64_t* src, uint64_t m, capy_hasher** out) {
  if (!out) return CAPY_ERR_BAD_ARG;
  *out = nullptr;
  if (hasher_check(ctx, h) || !hasher_portable(h) || (m && !src)) return CAPY_ERR_BAD_ARG;
  for (uint64_t j = 0; j < m; j++)
    if (src[j] >= h->n) return CAPY_ERR_BAD_ARG;  // (every m > 0 with n == 0 too)
  capy_hasher* f = nullptr;
  int rc = hasher_create(ctx, h->d_bits, h->kind, m, &f);
  if (rc) return rc;
  if (m) rc = fork_items(ctx, h, src, f);
  if (rc) {
    capy_hasher_free(f);
    return rc;
  }
  *out = f;
  return CAPY_OK;
}

void capy_hasher_free(capy_hasher* h) {
  if (!h) return;
  for (size_t k = 0; k < h->dev.size(); k++) {
    void* bufs[] = {h->d_state[k], h->d_carry[k], h->d_total[k], h->d_ks_state[k], h->d_ks_pos[k], h->d_h[k], h->d_bad[k],
                    h->d_state2[k], h->d_s[k], h->d_k[k], h->d_s_be[k], h->d_n1[k], h->d_state0[k], h->d_ks_state0[k],
                    h->d_verdict[k]};
    bool any = false;
    for (void* p : bufs) any = any || p;
    if (!any) continue;
    const size_t m = (size_t)hasher_items(h, (int)k);
    DeviceGuard g(h->dev[k]);
    cudaDeviceSynchronize();  // work still queued on a caller's stream may read them
    // after the key block a KMAC state is key material, and so is a keystream state: zeroed before the memory goes back
    if (h->d_state[k]) cudaMemset(h->d_state[k], 0, m * 200);
    if (h->d_carry[k]) cudaMemset(h->d_carry[k], 0, m * h->rate);
    if (h->d_ks_state[k]) cudaMemset(h->d_ks_state[k], 0, m * 200);
    // sign streams: s, k, the first "N" output and the second "N" state; decryption streams: the ke / ka states
    for (void* p : {(void*)h->d_state2[k], (void*)h->d_state0[k], (void*)h->d_ks_state0[k]})
      if (p) cudaMemset(p, 0, m * 200);
    for (void* p : {(void*)h->d_s[k], (void*)h->d_k[k], (void*)h->d_s_be[k], (void*)h->d_n1[k]})
      if (p) cudaMemset(p, 0, m * 56);
    cudaDeviceSynchronize();
    for (void* p : bufs)
      if (p) cudaFree(p);
  }
  delete h;
}

}  // extern "C"
