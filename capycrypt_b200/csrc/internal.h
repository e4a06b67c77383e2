// internal.h -- host-side context shared by the translation units of libcapycrypt_gpu.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <string_view>
#include <thread>
#include <vector>

#include "../../include/capy_gpu.h"
#include "sponge_job.h"

namespace capy {

constexpr int kNumStreams = 3;

// Device scratch slots.  Every internal stream has its own set of them (DeviceCtx::scratch[set][slot]): the chunks of a
// host call run on the three streams at once, and scratch_get picks the set from the stream, so two streams never share
// a buffer.  A caller's stream (the _dev entry points) uses set 0.
enum Slot {
  // device buffers of the inputs and outputs of a host entry point, handed out in declaration order by HostChunk
  // (hostbatch.h); only the scattered multi-device path of capy_sha3_batch names them.  Shared by all host entry points:
  // one host call holds a device at a time, waits for its streams and drains its staging before it returns, and no
  // device pipeline uses these slots.
  kHost0, kHost1, kHost2, kHost3, kHost4, kHost5, kHost6, kHost7,
  kFlag,                    // "bad point" flag of run_chunks (hostbatch.h)
  kPlanHist, kPlanOrder,    // plan_ragged: device length histogram (+ summary), work order
  kChainStates, kChainSync,  // chain hand-off of launch_sponge_chain / launch_chain_jobs: states, tickets
  // Ed448 pipelines (ed448_api.cu)
  kEdKWords, kEdSWords, kEdProj, kEdProj2, kEdBad, kEdTmp56A, kEdTmp56B, kEdTmp56C,
  kEdPubRep,                // a prepared key's point repeated n times (the fallback of the prepared entry points)
  // AE pipelines (ae_api.cu)
  kAeKeys, kAeKeyOff, kAeKeyMat, kAeTNew, kAeWx, kAeProj, kAeBad, kAeKw, kAeSk,
  kSlotsPerStream
};

// grow-only device scratch
struct Scratch {
  void* p = nullptr;
  size_t cap = 0;
};

struct PrefixState {
  uint64_t* d_state = nullptr;   // 25 lanes after the whole-block part of the prefix
  uint8_t* d_prefix = nullptr;   // prefix bytes on the device
  uint32_t prefix_len = 0;
  uint32_t skip_blocks = 0;
  uint64_t last_use = 0;         // LRU stamp (the customisation string is caller-controlled: the cache is bounded)
};
constexpr size_t kMaxPrefixEntries = 64;

// How a ragged batch is launched (sha3_api.cu: plan_ragged builds it, run_sponge follows it).  `order` = work order
// (longest first) or nullptr.
struct LaunchPlan {
  const uint32_t* order = nullptr;
  int warps_per_smsp = 0;   // 0 = unthrottled
  uint64_t warp_items[3] = {0, 0, 0};  // one warp per item: [c - 1] of them run c chains per scheduler (ranks in this order)
  uint64_t pair_items = 0;             // the next ranks: two threads per item
  uint64_t uniform_blocks = 0;         // != 0: every item holds this many whole blocks (+ a partial one): nothing to order,
                                       // and run_sponge may cut the chains
  // chain-bound batch: one launch of the warp, pair and thread tiers (sponge_tiered_kernel)
  bool tiered() const { return warp_items[0] || warp_items[1] || warp_items[2] || pair_items; }
};

// Cached plan of a ragged batch, keyed by the caller's offsets array (capy_gpu_set_plan_cache): a repeated call with the
// same (device pointer, n, unit) launches without touching the host.  A stale plan (the caller rewrote the offsets in
// place) costs speed only: `order` stays a permutation of [0, n) and any item may run in any tier.
struct PlanEntry {
  const uint64_t* off = nullptr;
  uint64_t n = 0;
  uint32_t unit = 0;
  bool allow_pair = true;
  LaunchPlan plan;
  uint32_t* owned_order = nullptr;
  uint64_t last_use = 0;
};
constexpr size_t kMaxPlanEntries = 16;

// persistent worker thread of one device of a multi-device ctx: host entry points post their per-device closure here
// instead of spawning a std::thread per call
class DeviceWorker {
 public:
  explicit DeviceWorker(int dev);
  ~DeviceWorker();
  void post(std::function<void()> f);

 private:
  void loop(int dev);
  std::mutex m_;
  std::condition_variable cv_;
  std::deque<std::function<void()>> q_;
  bool stop_ = false;
  std::thread th_;
};

struct Ed448Tables;  // defined in ed448_api.cu

// ---- staging of pageable host memory ---------------------------------------------------------------------------------
// A copy between the device and ordinary (pageable) host memory goes through the driver's own bounce buffers on the
// calling thread: 8.9 GB/s for the 64 MiB + 32 MiB of BASELINE config 1 against 46.7 GB/s from page-locked buffers.  Host
// entry points therefore stage large pageable buffers themselves: a few host threads copy a piece into (out of) a
// page-locked double buffer while the DMA of the previous piece runs.  Buffers from capy_host_alloc skip all of this.
constexpr size_t kStagePiece = 8ull << 20;      // bytes per staging half
constexpr size_t kStageMinBytes = 256ull << 10;  // smaller copies are left to the driver
struct StageSlot {
  uint8_t* p = nullptr;  // 2 x kStagePiece, page-locked
  cudaEvent_t ev[2] = {nullptr, nullptr};
  bool pending[2] = {false, false};
  // device-to-host: where the bytes of a half go once its copy has arrived
  void* drain_dst[2] = {nullptr, nullptr};
  size_t drain_bytes[2] = {0, 0};
  int next = 0;
};

// a few persistent helper threads that split one memcpy between them (and the caller)
class CopyPool {
 public:
  explicit CopyPool(int helpers);
  ~CopyPool();
  void copy(void* dst, const void* src, size_t bytes);

 private:
  void loop();
  std::mutex m_;
  std::condition_variable cv_, done_cv_;
  std::vector<std::thread> th_;
  uint8_t* dst_ = nullptr;
  const uint8_t* src_ = nullptr;
  size_t bytes_ = 0, slice_ = 0;
  int next_ = 0, slices_ = 0, left_ = 0;
  uint64_t gen_ = 0;
  bool stop_ = false;
};

struct DeviceCtx {
  int dev = 0;
  int index = 0;  // position in capy_ctx::devs
  cudaStream_t streams[kNumStreams] = {};
  Scratch scratch[kNumStreams][kSlotsPerStream];
  Scratch vb_slabs;  // per-SM table slabs of var_base_kernel: shared by all streams (an SM runs one var_base block at a time)
  std::map<std::string, PrefixState> prefix_cache;
  std::vector<PlanEntry> plans;
  // host copies of the offsets arrays a host entry point has staged into device scratch (HostChunk::in_packed), keyed by
  // the device address: plan_ragged reads the lengths from the host copy instead of fetching the histogram summary from
  // the device (no stream synchronisation inside a host-buffer call).  Valid only while that host call runs (HostOffScope).
  struct HostOff {
    const uint64_t* d_off;
    const uint64_t* h_off;
    uint64_t count;  // entries (items + 1)
  };
  std::vector<HostOff> host_offs;
  uint64_t use_clock = 0;
  Ed448Tables* ed = nullptr;
  int sm_count = 0;
  // host-side state of THIS device (scratch slots, caches, tables): one lock per device, so callers that use
  // different devices of a ctx do not serialise
  std::unique_ptr<std::mutex> mu{new std::mutex()};
  std::unique_ptr<DeviceWorker> worker;  // only in a multi-device ctx
  // staging of pageable host buffers, one double buffer per scratch slot that needs it (created at first use)
  StageSlot stage[kNumStreams][kSlotsPerStream];
  std::unique_ptr<CopyPool> copy_pool;
};

}  // namespace capy

struct capy_ctx {
  std::vector<capy::DeviceCtx> devs;
  std::mutex err_mu;  // guards last_cuda_error only
  std::string last_cuda_error;
  std::atomic<uint64_t> launches{0};
  std::atomic<int> plan_cache{0};
};

// A public key prepared for many operations (capy_ed448_pub_prepare, ed448_api.cu).  Owns, on every device of the ctx
// that prepared it, V's affine bytes and -- when V has order r -- the comb table of phi(V).
struct capy_ed448_pub {
  const capy_ctx* ctx = nullptr;
  uint8_t xy[112] = {};
  bool comb = false;
  std::vector<int> dev;            // CUDA device of every ctx device (frees without the ctx)
  std::vector<uint8_t*> d_xy;      // [device index] V's 112 affine bytes
  std::vector<uint32_t*> d_table;  // [device index] comb table of phi(V), or nullptr
};

// A batch of resumable SHA3-d / KMACXOF streams (capy_sha3_hasher_new / capy_kmac_xof_hasher_new, sha3_api.cu).  Items
// [first[k], first[k + 1]) live on device k of the ctx that created it, in buffers of their own: they are not scratch
// slots, so the one-shot calls between two updates never touch them.  On device k, item j (counted from first[k]) has
//   d_state[k]  25 lanes at [l * items_k + j]: every whole block of its stream so far (200 B per item)
//   d_carry[k]  the bytes behind the last whole block at [j * rate ..), total % rate of them
//   d_total[k]  [j] = message bytes absorbed so far (uint64)
// Encryption streams (capy_sponge_encrypt_stream_new / capy_ed448_key_encrypt_stream_new, ae_api.cu) are KMAC streams
// keyed by ka -- the tag -- with a keystream sponge beside each (SpongeSqueeze):
//   d_ks_state[k]  25 lanes at [l * items_k + j]: the keystream sponge at the start of its current squeeze block
//   d_ks_pos[k]    [j] = keystream bytes used so far
// Verification streams (capy_ed448_verify_stream_new, ed448_api.cu) are KMAC streams keyed by U'.x with S = "T", and keep
//   d_h[k]    [j * 56 ..) the signature's h ;  d_bad[k]  [j] = V_j is off the curve
namespace capy {
enum HasherKind { kSha3Stream, kKmacStream, kEncryptStream, kVerifyStream };
}
struct capy_hasher {
  const capy_ctx* ctx = nullptr;
  int d_bits = 0;
  int kind = capy::kSha3Stream;
  bool kmac = false;  // every kind but kSha3Stream
  uint32_t rate = 0;
  uint32_t tag_bits = 0;           // encryption and verification streams: the width of the final
  uint64_t n = 0;
  std::vector<uint64_t> first;     // [device index] first item; first[devices] = n
  std::vector<int> dev;            // CUDA device of every ctx device (frees without the ctx)
  std::vector<uint64_t*> d_state;  // [device index], nullptr when the device holds no item
  std::vector<uint8_t*> d_carry;
  std::vector<uint64_t*> d_total;
  std::vector<uint64_t*> d_ks_state;  // encryption streams only
  std::vector<uint64_t*> d_ks_pos;
  std::vector<uint8_t*> d_h;          // verification streams only
  std::vector<uint8_t*> d_bad;
  std::vector<char> finished;      // [device index] its items were finalised
};

namespace capy {

// RAII device switch
struct DeviceGuard {
  int prev = 0;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() { cudaSetDevice(prev); }
};

int cuda_fail(capy_ctx* ctx, cudaError_t e, const char* what);
#define CAPY_CUDA(ctx, expr)                                             \
  do {                                                                   \
    cudaError_t _e = (expr);                                             \
    if (_e != cudaSuccess) return ::capy::cuda_fail((ctx), _e, #expr);   \
  } while (0)

inline bool dev_index_ok(const capy_ctx* ctx, int dev_index) {
  return ctx && dev_index >= 0 && dev_index < (int)ctx->devs.size();
}
// The _dev entry points: checks ctx and dev_index, then holds the device's lock (host-side state of this device: scratch
// slots, caches, tables) and makes it current; defines `dc` and `st` (the caller's stream).
#define CAPY_DEV_PROLOGUE                                                                    \
  if (!dev_index_ok(ctx, dev_index)) return CAPY_ERR_BAD_ARG;                                \
  DeviceCtx& dc = ctx->devs[dev_index];                                                      \
  std::lock_guard<std::mutex> lk(*dc.mu);                                                    \
  DeviceGuard g(dc.dev);                                                                     \
  cudaStream_t st = (cudaStream_t)stream;

// k when st is the device's internal stream k; 0 for any other stream (a caller's stream)
inline int stream_set(const DeviceCtx& dc, cudaStream_t st) {
  for (int k = 1; k < kNumStreams; k++)
    if (dc.streams[k] == st) return k;
  return 0;
}

// grows `s` to at least `bytes`; returns nullptr on OOM
void* scratch_grow(Scratch& s, size_t bytes);
// the buffer of `slot` in the slot set of stream st; returns nullptr on OOM
inline void* scratch_get(DeviceCtx& dc, cudaStream_t st, Slot slot, size_t bytes) {
  return scratch_grow(dc.scratch[stream_set(dc, st)][slot], bytes);
}
#define CAPY_SCRATCH(var, type, slot, bytes)                    \
  type* var = (type*)scratch_get(dc, st, (slot), (bytes));      \
  if (!var) return CAPY_ERR_OOM;

inline unsigned grid_for(uint64_t n, unsigned block) { return (unsigned)((n + block - 1) / block); }

// host <-> device copies of the host entry points (hostbatch.h); `slot` = the scratch slot of the device buffer
int copy_in(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, Slot slot, void* d_dst, const void* h_src, size_t bytes);
int copy_out(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, Slot slot, void* h_dst, const void* d_src, size_t bytes);
// waits for the staged device-to-host copies of this device and hands their bytes to the caller's buffers
int stage_drain(capy_ctx* ctx, DeviceCtx& dc);
void stage_free(DeviceCtx& dc);

// the host arrays registered in dc.host_offs belong to the caller of ONE host entry point: forget them when it returns
struct HostOffScope {
  DeviceCtx& dc;
  explicit HostOffScope(DeviceCtx& d) : dc(d) { dc.host_offs.clear(); }
  ~HostOffScope() { dc.host_offs.clear(); }
};
inline void host_off_register(DeviceCtx& dc, const uint64_t* d_off, const uint64_t* h_off, uint64_t count) {
  for (auto& e : dc.host_offs)
    if (e.d_off == d_off) {
      e.h_off = h_off;
      e.count = count;
      return;
    }
  dc.host_offs.push_back({d_off, h_off, count});
}
inline const uint64_t* host_off_find(const DeviceCtx& dc, const uint64_t* d_off, uint64_t n) {
  for (const auto& e : dc.host_offs)
    if (e.d_off == d_off && e.count >= n + 1) return e.h_off;
  return nullptr;
}

inline bool valid_secparam(int d) { return d == 224 || d == 256 || d == 384 || d == 512; }

// ---- device-level launchers (async on `stream`), implemented in sha3_api.cu -----------------
// One KMACXOF pass over job.n items.  The caller fills in the per-item fields of `job`: keys, messages (none: data stays
// nullptr and msg_len 0), outputs, xor_in.  The launchers add the operator fields and the prefix of (d_bits, custom).
struct KmacPass {
  int d_bits;
  std::string_view custom;
  bool no_sort = false;  // keep the caller's order (skips the length bucketing and its tiny D2H sync)
  SpongeJob job{};
  KmacPass(int d, std::string_view s, uint64_t n) : d_bits(d), custom(s) { job.n = n; }
};
int launch_kmac_xof(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& a);
// two passes over the same items (same d, same n) as one launch; the plan (work order) is taken from `a`
int launch_kmac_xof2(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& a, const KmacPass& b);
// two passes where `second` absorbs what `first` wrote for the same item: one launch of dependent jobs when the batch is large
int launch_kmac_xof_dep(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& first, const KmacPass& second);
// The state of a KMAC pass without message (a.job: keys, n) before its first squeeze, stored at states[l * n + i]: with
// the trailer, after P | KB | 00 01 04 | pad (a keystream at position 0); without, exactly after P | KB (the start of a
// KMAC stream)
int launch_kmac_state(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream, const KmacPass& a, bool trailer, uint64_t* states);
// a stream batch of `kind` (HasherKind) with zeroed buffers on every device that holds items (blocking; sha3_api.cu)
int hasher_create(capy_ctx* ctx, int d_bits, int kind, uint64_t n, capy_hasher** out, uint32_t tag_bits = 0);
// ok[i] = (hp_i == h_i) && !bad[i] over 56-byte rows; *bad_flag |= 1 when a bad[i] is set (ed448_api.cu)
int launch_verify_compare(capy_ctx* ctx, cudaStream_t st, const uint8_t* hp, const uint8_t* h, const uint8_t* bad, uint8_t* ok,
                          int* bad_flag, uint64_t n);

}  // namespace capy
