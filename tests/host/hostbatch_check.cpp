// tests/host/hostbatch_check.cpp -- CPU check of the host-side batch plumbing (capycrypt_b200/csrc/hostbatch.h):
// shard/chunk boundaries of split_items, the chunk counts of fixed and ragged batches, and the staging of one chunk
// (HostChunk) against host-memory stand-ins for device scratch and copies.  Compiled with g++ against the CUDA headers
// only (nothing here touches a device); run by tests/test_hostbatch.py.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include "../../capycrypt_b200/csrc/hostbatch.h"
using namespace capy;

// stand-ins for ctx.cu: scratch in host memory, copies as memcpy; copy_out records the slot of every output it copies
static std::vector<Slot> g_out_slots;
namespace capy {
void* scratch_grow(Scratch& s, size_t bytes) {
  if (s.cap < bytes) {
    free(s.p);
    s.p = malloc(bytes);
    s.cap = bytes;
  }
  return s.p;
}
int copy_in(capy_ctx*, DeviceCtx&, cudaStream_t, Slot, void* d_dst, const void* h_src, size_t bytes) {
  memcpy(d_dst, h_src, bytes);
  return CAPY_OK;
}
int copy_out(capy_ctx*, DeviceCtx&, cudaStream_t, Slot slot, void* h_dst, const void* d_src, size_t bytes) {
  g_out_slots.push_back(slot);
  memcpy(h_dst, d_src, bytes);
  return CAPY_OK;
}
DeviceWorker::~DeviceWorker() {}
CopyPool::~CopyPool() {}
}  // namespace capy

#define EXPECT(c) do { if (!(c)) { printf("FAIL line %d: %s\n", __LINE__, #c); return 1; } } while (0)

static bool covers(const std::vector<Range>& r, uint64_t i0, uint64_t i1) {
  uint64_t at = i0;
  for (const Range& x : r) {
    if (x.i0 != at || x.i1 <= x.i0) return false;
    at = x.i1;
  }
  return at == i1;
}

int main() {
  // fixed-size items: equal parts, contiguous, complete
  auto r = split_items(nullptr, 64, 0, 1000, 8, 0);
  EXPECT(r.size() == 8 && covers(r, 0, 1000));
  for (const Range& x : r) EXPECT(x.i1 - x.i0 == 125);
  // more parts than items, empty range, sub-range
  EXPECT(split_items(nullptr, 64, 0, 3, 8, 0).size() == 3);
  EXPECT(split_items(nullptr, 64, 5, 5, 4, 0).empty());
  EXPECT(covers(split_items(nullptr, 1, 10, 20, 3, 0), 10, 20));
  // ragged items are balanced by bytes (+ a per-item cost): one 1 MB item against 1000 small ones
  std::vector<uint64_t> off(1002, 0);
  off[1] = 1000000;
  for (int i = 2; i <= 1001; i++) off[i] = off[i - 1] + 1000;
  r = split_items(off.data(), 0, 0, 1001, 2, 0);
  EXPECT(r.size() == 2 && covers(r, 0, 1001) && r[0].i1 == 1);  // the big item alone is half of the bytes
  // zero-length items everywhere: falls back to the per-item cost
  std::vector<uint64_t> zeros(101, 0);
  r = split_items(zeros.data(), 0, 0, 100, 4, 200);
  EXPECT(r.size() == 4 && covers(r, 0, 100));
  // chunk counts: 8 MiB chunks, never fewer than 1024 items per chunk
  EXPECT(chunk_count(64ull << 20, 1 << 20) == 8);
  EXPECT(chunk_count(1, 1) == 1);
  EXPECT(chunk_count(1ull << 30, 2048) == 2);
  // ragged: a chunk must hold ~8192 x its longest message, so long messages mean few chunks
  std::vector<uint64_t> big(3001, 0);
  for (int i = 1; i <= 3000; i++) big[i] = big[i - 1] + (1u << 20);  // 3000 x 1 MiB = 2.9 GiB
  EXPECT(ragged_chunk_count(big.data(), 0, 3000, 0) == 1);
  std::vector<uint64_t> small(1 << 20 | 1, 0);
  for (size_t i = 1; i < small.size(); i++) small[i] = small[i - 1] + 64;  // 2^20 x 64 B
  EXPECT(ragged_chunk_count(small.data(), 0, 1 << 20, 0) == 8);
  // ---- LPT shares of a ragged batch over several devices ----
  {
    // a batch sorted by length, longest first: a contiguous split by bytes gives device 0 all the long chains
    std::vector<uint64_t> so(1 + 40 + 100000, 0);
    for (int i = 1; i <= 40; i++) so[i] = so[i - 1] + (1u << 20);
    for (size_t i = 41; i < so.size(); i++) so[i] = so[i - 1] + 400;
    const uint64_t n = so.size() - 1;
    for (size_t parts : {2, 4, 8}) {
      auto sh = lpt_shares(so.data(), n, parts, 72, 2);
      EXPECT(sh.size() == parts);
      std::vector<int> seen(n, 0);
      uint64_t max_cost = 0, sum_cost = 0, max_long = 0, min_long = ~0ull;
      for (const DeviceShare& d : sh) {
        uint64_t prev = 0, longs = 0, items = 0;
        for (const Run& r : d.runs) {
          EXPECT(r.i0 < r.i1 && r.i0 >= prev);  // increasing, non-overlapping
          prev = r.i1;
          for (uint64_t i = r.i0; i < r.i1; i++) { seen[i]++; items++; if (i < 40) longs++; }
        }
        EXPECT(items == d.items);
        max_cost = std::max(max_cost, d.cost);
        sum_cost += d.cost;
        max_long = std::max(max_long, longs);
        min_long = std::min(min_long, longs);
        EXPECT(d.runs.size() <= 64);  // a handful of copies per device, not one per message
      }
      for (uint64_t i = 0; i < n; i++) EXPECT(seen[i] == 1);  // a partition
      EXPECT(max_long - min_long <= 1);                        // the long chains are dealt out evenly
      EXPECT(max_cost * parts <= sum_cost + sum_cost / 20 + parts * 15000);  // and the total work is balanced
    }
    // uniform batch: no outliers -> plain contiguous ranges, one run per device
    auto sh = lpt_shares(small.data(), 1 << 20, 4, 136, 1);
    for (const DeviceShare& d : sh) EXPECT(d.runs.size() == 1 && d.items == (1u << 18));
    // fewer items than devices, empty batch
    EXPECT(lpt_shares(so.data(), 3, 8, 72, 2).size() == 3);
    EXPECT(lpt_shares(so.data(), 0, 4, 72, 2).size() == 1);
  }
  // ---- HostChunk: every declaration takes the next kHost slot; outputs come back in declaration order ----
  {
    capy_ctx ctx;
    DeviceCtx dc;
    cudaStream_t st = dc.streams[0];
    Scratch* slots = dc.scratch[stream_set(dc, st)];
    std::vector<uint64_t> po(41, 0);  // 40 packed items of 0..12 bytes: item 10 starts off a 16-byte boundary
    for (int i = 1; i <= 40; i++) po[i] = po[i - 1] + (uint64_t)(i * 7 % 13);
    std::vector<uint8_t> packed(po[40]), rows(40 * 56);
    for (size_t i = 0; i < packed.size(); i++) packed[i] = (uint8_t)(i * 31 + 7);
    for (size_t i = 0; i < rows.size(); i++) rows[i] = (uint8_t)(i * 13 + 1);
    const Range r{10, 30};
    EXPECT(po[r.i0] % 16 != 0);
    HostChunk io(&ctx, dc, st, r, nullptr);
    EXPECT(io.n() == 20 && io.i0() == 10 && io.i1() == 30 && io.d_flag() == nullptr);
    const StagedPacked sp = io.in_packed(packed.data(), po.data());
    const uint8_t* d_rows = io.in(rows.data(), 56);
    std::vector<uint8_t> h_rows(40 * 7, 0xee), h_packed(po[40], 0xee);
    uint8_t* d_out = io.out(h_rows.data(), 7);
    uint8_t* d_pk = io.out_packed(h_packed.data(), po.data());
    EXPECT(io.rc() == CAPY_OK && sp.d_base && d_rows && d_out && d_pk);
    // slots in declaration order: packed data, its offsets, the rows, then the two outputs
    const uint64_t a0 = po[r.i0] & ~(uint64_t)15;
    EXPECT(sp.d_base + a0 == slots[kHost0].p && (const void*)sp.d_off == slots[kHost1].p);
    EXPECT(d_rows == slots[kHost2].p && d_out == slots[kHost3].p && d_pk + a0 == slots[kHost4].p);
    EXPECT(slots[kHost0].cap == po[r.i1] - a0 + 16 && slots[kHost1].cap == 21 * 8 && slots[kHost2].cap == 20 * 56 + 16);
    for (uint64_t i = r.i0; i <= r.i1; i++) EXPECT(sp.d_off[i - r.i0] == po[i]);
    EXPECT(memcmp(sp.d_base + po[r.i0], packed.data() + po[r.i0], po[r.i1] - po[r.i0]) == 0);
    EXPECT(memcmp(d_rows, rows.data() + 56 * r.i0, 20 * 56) == 0);
    EXPECT(host_off_find(dc, sp.d_off, 20) == po.data() + r.i0);  // plan_ragged may plan from the caller's offsets
    // the pipeline writes the outputs; copy_back hands exactly the chunk's bytes to the caller's buffers
    for (int k = 0; k < 20 * 7; k++) d_out[k] = (uint8_t)k;
    for (uint64_t b = po[r.i0]; b < po[r.i1]; b++) d_pk[b] = (uint8_t)(b ^ 0x5a);
    EXPECT(io.copy_back() == CAPY_OK);
    EXPECT(g_out_slots.size() == 2 && g_out_slots[0] == kHost3 && g_out_slots[1] == kHost4);
    for (size_t k = 0; k < h_rows.size(); k++)
      EXPECT(h_rows[k] == (k >= 7 * r.i0 && k < 7 * r.i1 ? (uint8_t)(k - 7 * r.i0) : 0xee));
    for (uint64_t b = 0; b < h_packed.size(); b++)
      EXPECT(h_packed[b] == (b >= po[r.i0] && b < po[r.i1] ? (uint8_t)(b ^ 0x5a) : 0xee));
    // a declaration past kHost7 fails instead of reusing a slot, and so does everything after it
    HostChunk full(&ctx, dc, st, r, nullptr);
    for (int k = kHost0; k <= kHost7; k++) EXPECT(full.in(rows.data(), 1) != nullptr);
    EXPECT(full.rc() == CAPY_OK);
    EXPECT(full.out(h_rows.data(), 7) == nullptr && full.rc() == CAPY_ERR_BAD_ARG);
    EXPECT(full.in(rows.data(), 1) == nullptr && full.copy_back() == CAPY_ERR_BAD_ARG);
  }
  printf("hostbatch ok\n");
  return 0;
}
