// hostbatch.h -- host-buffer plumbing shared by the SHA3, Ed448 and AE entry points.
#pragma once
#include <algorithm>
#include <condition_variable>
#include <mutex>
#include <vector>

#include "internal.h"

namespace capy {

// ---- host-buffer plumbing -----------------------------------------------------------------------
// Splits items [0, n) across the ctx devices (contiguous ranges, balanced by bytes) and, inside a
// device, into chunks that are copied in, processed and copied out on rotating streams so that
// H2D, kernel and D2H of neighbouring chunks overlap.  No collective: items are independent.
struct Range {
  uint64_t i0, i1;
};

inline std::vector<Range> split_items(const uint64_t* off, uint64_t fixed_len, uint64_t i0, uint64_t i1, size_t parts,
                                      uint64_t per_item_cost) {
  std::vector<Range> r;
  if (i1 <= i0) return r;
  parts = std::max<size_t>(1, std::min<uint64_t>(parts, i1 - i0));
  auto cost_at = [&](uint64_t i) -> uint64_t {  // cumulative cost of items [i0, i)
    uint64_t bytes = off ? off[i] - off[i0] : (i - i0) * fixed_len;
    return bytes + (i - i0) * per_item_cost;
  };
  const uint64_t total = cost_at(i1);
  uint64_t start = i0;
  for (size_t p = 1; p <= parts && start < i1; p++) {
    uint64_t end;
    if (p == parts) {
      end = i1;
    } else {
      const uint64_t target = total / parts * p;
      uint64_t lo = start + 1, hi = i1;
      while (lo < hi) {  // first index with cumulative cost >= target
        uint64_t mid = (lo + hi) / 2;
        if (cost_at(mid) < target) lo = mid + 1;
        else hi = mid;
      }
      end = lo;
    }
    if (end > start) r.push_back({start, end});
    start = end;
  }
  return r;
}

// ---- ragged sponge batches over several devices: longest-processing-time-first over the chains (SURVEY.md 8e) --------
// A sponge is sequential per message, so a device cannot finish before its longest message has, and a contiguous split
// by bytes can hand one device most of the long chains (a batch sorted by length does).  The outliers -- messages that
// cost at least 8 x the average, at most kLptMaxLong of them -- are dealt out longest first, each to the device with
// the least work so far (LPT); the remaining messages follow in contiguous index ranges that top every device up to the
// same load, so the bulk of the batch still moves with one copy per range.  A device's share is a list of runs of
// consecutive items in increasing index order.
struct Run {
  uint64_t i0, i1;
};
struct DeviceShare {
  std::vector<Run> runs;
  uint64_t items = 0, bytes = 0, cost = 0;
};
constexpr size_t kLptMaxLong = 4096;

inline std::vector<DeviceShare> lpt_shares(const uint64_t* off, uint64_t n, size_t parts, uint32_t unit_bytes,
                                           uint64_t per_item_cost) {
  parts = std::max<size_t>(1, std::min<uint64_t>(parts, std::max<uint64_t>(n, 1)));
  std::vector<DeviceShare> sh(parts);
  if (n == 0) return sh;
  auto cost_of = [&](uint64_t i) -> uint64_t { return (off[i + 1] - off[i]) / unit_bytes + per_item_cost; };
  uint64_t total = 0;
  for (uint64_t i = 0; i < n; i++) total += cost_of(i);
  // outliers: cost >= 8 x average (only then can a single chain matter for the balance)
  const uint64_t thr = std::max<uint64_t>(8 * (total / n), per_item_cost + 1);
  std::vector<std::pair<uint64_t, uint64_t>> longs;  // (cost, index)
  if (parts > 1)
    for (uint64_t i = 0; i < n; i++) {
      const uint64_t c = cost_of(i);
      if (c >= thr) longs.emplace_back(c, i);
    }
  std::sort(longs.begin(), longs.end(), [](const auto& a, const auto& b) { return a.first != b.first ? a.first > b.first : a.second < b.second; });
  if (longs.size() > kLptMaxLong) longs.resize(kLptMaxLong);
  std::vector<uint64_t> load(parts, 0);
  std::vector<std::pair<uint64_t, uint32_t>> owner;  // (index, device) of the dealt-out items, sorted by index below
  owner.reserve(longs.size());
  for (const auto& l : longs) {
    size_t best = 0;
    for (size_t d = 1; d < parts; d++)
      if (load[d] < load[best]) best = d;
    load[best] += l.first;
    owner.emplace_back(l.second, (uint32_t)best);
  }
  std::sort(owner.begin(), owner.end());
  // everything else: contiguous ranges, every device topped up to total / parts
  auto push = [&](size_t d, uint64_t i) {
    DeviceShare& s = sh[d];
    if (!s.runs.empty() && s.runs.back().i1 == i) s.runs.back().i1 = i + 1;
    else s.runs.push_back({i, i + 1});
    s.items++;
    s.bytes += off[i + 1] - off[i];
    s.cost += cost_of(i);
  };
  // short-item budget of every device: what it lacks to total / parts, rescaled so that the budgets add up to the
  // cost of the short items; device d takes the short items whose running cost falls into its slice of that sum
  uint64_t long_total = 0;
  for (uint64_t l : load) long_total += l;
  const double rest = (double)(total - long_total), target = (double)total / (double)parts;
  std::vector<double> bound(parts);
  double lack = 0;
  for (size_t d = 0; d < parts; d++) lack += std::max(0.0, target - (double)load[d]);
  double accb = 0;
  for (size_t d = 0; d < parts; d++) {
    accb += lack > 0 ? std::max(0.0, target - (double)load[d]) * rest / lack : rest / (double)parts;
    bound[d] = accb;
  }
  size_t cur = 0, next_long = 0;
  double acc = 0;
  for (uint64_t i = 0; i < n; i++) {
    if (next_long < owner.size() && owner[next_long].first == i) {
      push(owner[next_long].second, i);
      next_long++;
      continue;
    }
    while (cur + 1 < parts && acc >= bound[cur]) cur++;
    push(cur, i);
    acc += (double)cost_of(i);
  }
  return sh;
}

// Runs fn(device, shard, bad_point) for every shard: inline on the caller's thread for a single shard, else on the
// devices' persistent worker threads (DeviceWorker), each holding its device's lock for the duration of its closure.
// fn may set *bad_point (an input point was not on the curve): the call then returns CAPY_ERR_BAD_POINT, unless a device
// failed otherwise, and only after every device has handed its outputs to the caller's buffers.
template <class F>
inline int for_each_device(capy_ctx* ctx, const std::vector<Range>& shards, F&& fn) {
  if (shards.empty()) return CAPY_OK;
  std::vector<int> rcs(shards.size(), CAPY_OK), bad(shards.size(), 0);
  if (shards.size() == 1) {
    DeviceCtx& dc = ctx->devs[0];
    std::lock_guard<std::mutex> lk(*dc.mu);
    DeviceGuard g(dc.dev);
    HostOffScope hs(dc);
    rcs[0] = fn(dc, shards[0], &bad[0]);
    const int rd = stage_drain(ctx, dc);  // staged device-to-host copies: hand the bytes to the caller's buffers
    if (!rcs[0]) rcs[0] = rd;
  } else {
    std::mutex m;
    std::condition_variable cv;
    size_t pending = shards.size();
    for (size_t k = 0; k < shards.size(); k++) {
      DeviceCtx& dc = ctx->devs[k];
      dc.worker->post([&, k] {
        {
          std::lock_guard<std::mutex> lk(*ctx->devs[k].mu);
          HostOffScope hs(ctx->devs[k]);
          rcs[k] = fn(ctx->devs[k], shards[k], &bad[k]);
          const int rd = stage_drain(ctx, ctx->devs[k]);
          if (!rcs[k]) rcs[k] = rd;
        }
        std::lock_guard<std::mutex> lk(m);
        if (--pending == 0) cv.notify_one();
      });
    }
    std::unique_lock<std::mutex> lk(m);
    cv.wait(lk, [&] { return pending == 0; });
  }
  for (int rc : rcs)
    if (rc) return rc;
  for (int b : bad)
    if (b) return CAPY_ERR_BAD_POINT;
  return CAPY_OK;
}

// Runs body(stream, chunk, d_flag) for the chunks of one device's shard, rotating over the device's internal streams, then
// waits for the streams it used.  body enqueues the copies in, the pipeline and the copies out of its chunk and does not
// wait, so the copies of one chunk run under the kernels of its neighbours.  With bad_flag_out, every stream's kFlag is
// zeroed first and passed as d_flag (else nullptr), and *bad_flag_out gets the OR of what the chunks left there.
template <class F>
inline int run_chunks(capy_ctx* ctx, DeviceCtx& dc, const std::vector<Range>& chunks, int* bad_flag_out, F&& body) {
  const int used = (int)std::min<size_t>(chunks.size(), kNumStreams);
  int* d_flags[kNumStreams] = {};
  if (bad_flag_out)
    for (int s = 0; s < used; s++) {
      d_flags[s] = (int*)scratch_get(dc, dc.streams[s], kFlag, sizeof(int));
      if (!d_flags[s]) return CAPY_ERR_OOM;
      CAPY_CUDA(ctx, cudaMemsetAsync(d_flags[s], 0, sizeof(int), dc.streams[s]));
    }
  for (size_t c = 0; c < chunks.size(); c++) {
    const int s = (int)(c % kNumStreams);
    const int rc = body(dc.streams[s], chunks[c], d_flags[s]);
    if (rc) return rc;
  }
  int h_flags[kNumStreams] = {};
  for (int s = 0; s < used; s++) {
    if (bad_flag_out) CAPY_CUDA(ctx, cudaMemcpyAsync(&h_flags[s], d_flags[s], sizeof(int), cudaMemcpyDeviceToHost, dc.streams[s]));
    CAPY_CUDA(ctx, cudaStreamSynchronize(dc.streams[s]));
  }
  if (bad_flag_out)
    for (int s = 0; s < used; s++) *bad_flag_out |= h_flags[s];
  return CAPY_OK;
}

// one packed host input staged per chunk: bytes [a0, off[i1]) with a0 = off[i0] rounded down to 16
struct StagedPacked {
  const uint8_t* d_base = nullptr;  // device pointer such that d_base + off[i] addresses item i
  const uint64_t* d_off = nullptr;  // device copy of off[i0 .. i1]
};

// The device buffers of one chunk's inputs and outputs (run_host_call).  Every declaration takes the next kHost slot, so
// two buffers of one call never share one, and a declaration past kHost7 is an error rather than a wrap-around.  Inputs
// are copied in when declared; outputs are copied back to the caller's buffers, in the order declared, by copy_back.  A
// failed declaration returns nullptr and makes rc() nonzero; the declarations after it do nothing.
class HostChunk {
 public:
  HostChunk(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, Range r, int* d_flag)
      : ctx_(ctx), dc_(dc), st_(st), r_(r), d_flag_(d_flag) {}
  uint64_t i0() const { return r_.i0; }
  uint64_t i1() const { return r_.i1; }
  uint64_t n() const { return r_.i1 - r_.i0; }
  int* d_flag() const { return d_flag_; }  // run_chunks' bad-point flag of this stream, or nullptr
  int rc() const { return rc_; }

  // n() rows of `row` bytes from host + row * i0 (`bytes` overrides the length, e.g. a short last row); 16 bytes of slack
  const uint8_t* in(const void* host, size_t row, size_t bytes = ~size_t(0)) {
    if (bytes == ~size_t(0)) bytes = row * n();
    Slot s{};
    uint8_t* d = grab(bytes + 16, &s);
    if (d) note(copy_in(ctx_, dc_, st_, s, d, (const uint8_t*)host + row * r_.i0, bytes));
    return rc_ ? nullptr : d;
  }

  // the items [i0, i1) of a packed input: bytes [a0, off[i1]) with a0 = off[i0] rounded down to 16, and off[i0 .. i1]
  StagedPacked in_packed(const uint8_t* data, const uint64_t* off) {
    const uint64_t a0 = off[r_.i0] & ~(uint64_t)15;
    const size_t bytes = (size_t)(off[r_.i1] - a0), count = (size_t)n() + 1;
    Slot sd{}, so{};
    uint8_t* d_data = grab(bytes + 16, &sd);
    uint64_t* d_off = (uint64_t*)grab(count * 8, &so);
    if (!rc_) note(copy_in(ctx_, dc_, st_, sd, d_data, data + a0, bytes));
    if (!rc_) note(copy_in(ctx_, dc_, st_, so, d_off, off + r_.i0, count * 8));
    if (rc_) return {};
    host_off_register(dc_, d_off, off + r_.i0, count);  // plan_ragged plans from the host copy: no device round trip
    return {rebase(d_data, a0), d_off};
  }

  // n() rows of `row` bytes, copied back to host + row * i0
  uint8_t* out(void* host, size_t row) {
    Slot s{};
    uint8_t* d = grab(row * n(), &s);
    if (d) outs_.push_back({s, (uint8_t*)host + row * r_.i0, d, row * n()});
    return d;
  }

  // the items [i0, i1) of a packed output: d + off[i] addresses item i (laid out as in_packed); bytes [off[i0], off[i1])
  // are copied back to the same offsets of host
  uint8_t* out_packed(uint8_t* host, const uint64_t* off) {
    const uint64_t a0 = off[r_.i0] & ~(uint64_t)15, b0 = off[r_.i0], b1 = off[r_.i1];
    Slot s{};
    uint8_t* d = grab((size_t)(b1 - a0) + 16, &s);
    if (!d) return nullptr;
    uint8_t* base = rebase(d, a0);
    outs_.push_back({s, host + b0, base + b0, (size_t)(b1 - b0)});
    return base;
  }

  // enqueues the copies of the outputs back to the caller's buffers (copy_out: pageable ones are staged)
  int copy_back() {
    if (rc_) return rc_;
    for (const Out& o : outs_) {
      const int rc = copy_out(ctx_, dc_, st_, o.slot, o.host, o.dev, o.bytes);
      if (rc) return rc;
    }
    return CAPY_OK;
  }

 private:
  struct Out {
    Slot slot;
    void* host;
    const uint8_t* dev;
    size_t bytes;
  };
  uint8_t* grab(size_t bytes, Slot* slot) {
    if (rc_) return nullptr;
    if (next_ > kHost7 - kHost0) {
      rc_ = CAPY_ERR_BAD_ARG;
      return nullptr;
    }
    *slot = (Slot)(kHost0 + next_++);
    uint8_t* d = (uint8_t*)scratch_get(dc_, st_, *slot, bytes);
    if (!d) rc_ = CAPY_ERR_OOM;
    return d;
  }
  void note(int rc) {
    if (!rc_) rc_ = rc;
  }
  static uint8_t* rebase(uint8_t* d, uint64_t a0) {
    return reinterpret_cast<uint8_t*>(reinterpret_cast<uintptr_t>(d) - (uintptr_t)a0);
  }
  capy_ctx* ctx_;
  DeviceCtx& dc_;
  cudaStream_t st_;
  Range r_;
  int* d_flag_;
  int next_ = 0, rc_ = CAPY_OK;
  std::vector<Out> outs_;
};

// One host call: the shards go to the ctx devices (for_each_device), chunks_of_shard(shard) cuts a shard into the chunks
// that rotate over the device's streams (run_chunks), and body(dc, st, io) declares a chunk's inputs and outputs on `io`
// and enqueues its pipeline; the outputs are then copied back.  With bad_points the chunks get run_chunks' bad-point
// flag (io.d_flag()), and a bad point anywhere makes the call return CAPY_ERR_BAD_POINT.
template <class Chunks, class Body>
inline int run_host_call(capy_ctx* ctx, const std::vector<Range>& shards, Chunks&& chunks_of_shard, bool bad_points,
                         Body&& body) {
  return for_each_device(ctx, shards, [&](DeviceCtx& dc, Range sh, int* bad_point) -> int {
    return run_chunks(ctx, dc, chunks_of_shard(sh), bad_points ? bad_point : nullptr,
                      [&](cudaStream_t st, Range ch, int* d_flag) -> int {
                        HostChunk io(ctx, dc, st, ch, d_flag);
                        const int rc = body(dc, st, io);
                        return rc ? rc : io.copy_back();
                      });
  });
}

// the chunker of the calls that run a device's shard as one chunk
inline std::vector<Range> one_chunk(Range sh) { return {sh}; }

constexpr uint64_t kChunkBytes = 8ull << 20;

// Ragged batches: a chunk is one launch, and a launch cannot finish before the longest message in it has (a sponge
// is sequential per message: ~30 ns per byte even with a whole warp on it), so a chunk that holds a long message must
// also hold enough other work to fill the GPU for that time (~270 GB/s): at least ~8192 x the longest message.
// Chunking a batch with 1 MiB messages into 8 MiB pieces made every piece chain-bound (measured: 6.9 s for 2.8 GiB).
inline size_t chunk_count(uint64_t bytes, uint64_t items);
inline size_t ragged_chunk_count(const uint64_t* off, uint64_t i0, uint64_t i1, uint64_t extra_bytes) {
  uint64_t max_len = 0;
  for (uint64_t i = i0; i < i1; i++) max_len = std::max<uint64_t>(max_len, off[i + 1] - off[i]);
  const uint64_t bytes = off[i1] - off[i0] + extra_bytes;
  const uint64_t min_chunk = std::max<uint64_t>(8ull << 20, 8192ull * max_len);
  const size_t by_size = (size_t)std::max<uint64_t>(1, bytes / min_chunk);
  return std::min<size_t>(by_size, chunk_count(bytes, i1 - i0));
}

inline size_t chunk_count(uint64_t bytes, uint64_t items) {
  uint64_t c = (bytes + kChunkBytes - 1) / kChunkBytes;
  c = std::max<uint64_t>(c, 1);
  c = std::min<uint64_t>(c, std::max<uint64_t>(items / 1024, 1));
  return (size_t)c;
}


}  // namespace capy
