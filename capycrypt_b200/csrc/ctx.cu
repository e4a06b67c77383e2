// ctx.cu -- context, streams, scratch memory and error plumbing of libcapycrypt_gpu.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "internal.h"

namespace capy {

int cuda_fail(capy_ctx* ctx, cudaError_t e, const char* what) {
  if (ctx) {
    std::lock_guard<std::mutex> lk(ctx->err_mu);
    ctx->last_cuda_error = std::string(cudaGetErrorName(e)) + ": " + cudaGetErrorString(e) + " at " + what;
  }
  cudaGetLastError();  // clear sticky-less errors
  return e == cudaErrorMemoryAllocation ? CAPY_ERR_OOM : CAPY_ERR_CUDA;
}

void* scratch_grow(Scratch& s, size_t bytes) {
  if (bytes == 0) bytes = 16;
  if (s.cap >= bytes) return s.p;
  if (s.p) {
    // other streams may still read the old buffer
    cudaDeviceSynchronize();
    cudaFree(s.p);
    s.p = nullptr;
    s.cap = 0;
  }
  size_t cap = (bytes + (bytes >> 2) + 255) & ~(size_t)255;  // 25% slack, 256-byte granules
  if (cudaMalloc(&s.p, cap) != cudaSuccess) {
    cudaGetLastError();
    if (cudaMalloc(&s.p, (bytes + 255) & ~(size_t)255) != cudaSuccess) {
      cudaGetLastError();
      s.p = nullptr;
      return nullptr;
    }
    cap = (bytes + 255) & ~(size_t)255;
  }
  s.cap = cap;
  return s.p;
}

void ed448_tables_free(DeviceCtx& dc);  // ed448_fixed.cu

DeviceWorker::DeviceWorker(int dev) { th_ = std::thread([this, dev] { loop(dev); }); }
DeviceWorker::~DeviceWorker() {
  {
    std::lock_guard<std::mutex> lk(m_);
    stop_ = true;
  }
  cv_.notify_all();
  if (th_.joinable()) th_.join();
}
void DeviceWorker::post(std::function<void()> f) {
  {
    std::lock_guard<std::mutex> lk(m_);
    q_.push_back(std::move(f));
  }
  cv_.notify_one();
}
void DeviceWorker::loop(int dev) {
  cudaSetDevice(dev);
  for (;;) {
    std::function<void()> f;
    {
      std::unique_lock<std::mutex> lk(m_);
      cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
      if (q_.empty()) return;  // stop requested and nothing left to run
      f = std::move(q_.front());
      q_.pop_front();
    }
    f();
  }
}

// ---- staging of pageable host buffers (internal.h) --------------------------------------------------------------------
CopyPool::CopyPool(int helpers) {
  for (int k = 0; k < helpers; k++) th_.emplace_back([this] { loop(); });
}
CopyPool::~CopyPool() {
  {
    std::lock_guard<std::mutex> lk(m_);
    stop_ = true;
  }
  cv_.notify_all();
  for (auto& t : th_)
    if (t.joinable()) t.join();
}
void CopyPool::loop() {
  uint64_t seen = 0;
  for (;;) {
    std::unique_lock<std::mutex> lk(m_);
    cv_.wait(lk, [&] { return stop_ || gen_ != seen; });
    if (stop_) return;
    seen = gen_;
    while (next_ < slices_) {
      const int k = next_++;
      const size_t a = (size_t)k * slice_, b = std::min(bytes_, a + slice_);
      lk.unlock();
      if (b > a) memcpy(dst_ + a, src_ + a, b - a);
      lk.lock();
      if (--left_ == 0) done_cv_.notify_all();
    }
  }
}
void CopyPool::copy(void* dst, const void* src, size_t bytes) {
  if (bytes < (1u << 20) || th_.empty()) {
    memcpy(dst, src, bytes);
    return;
  }
  std::unique_lock<std::mutex> lk(m_);
  dst_ = (uint8_t*)dst;
  src_ = (const uint8_t*)src;
  bytes_ = bytes;
  slices_ = (int)th_.size() + 1;
  slice_ = ((bytes + slices_ - 1) / slices_ + 4095) & ~(size_t)4095;
  next_ = 0;
  left_ = slices_;
  gen_++;
  cv_.notify_all();
  while (next_ < slices_) {  // the caller takes slices too
    const int k = next_++;
    const size_t a = (size_t)k * slice_, b = std::min(bytes_, a + slice_);
    lk.unlock();
    if (b > a) memcpy(dst_ + a, src_ + a, b - a);
    lk.lock();
    --left_;
  }
  done_cv_.wait(lk, [&] { return left_ == 0; });
}

static bool host_is_pageable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return a.type == cudaMemoryTypeUnregistered;
}

static int stage_ready(capy_ctx* ctx, DeviceCtx& dc, StageSlot& ss) {
  if (!ss.p) {
    void* p = nullptr;
    CAPY_CUDA(ctx, cudaHostAlloc(&p, 2 * kStagePiece, cudaHostAllocPortable));
    ss.p = (uint8_t*)p;
    for (int h = 0; h < 2; h++) CAPY_CUDA(ctx, cudaEventCreateWithFlags(&ss.ev[h], cudaEventDisableTiming));
  }
  if (!dc.copy_pool) {
    // one memcpy thread moves ~6-8 GB/s on this class of host; the link takes 52: up to seven helpers beside the caller,
    // fewer on small hosts (CAPY_COPY_THREADS overrides)
    int helpers = (int)std::thread::hardware_concurrency() / 2 - 1;
    if (const char* e = getenv("CAPY_COPY_THREADS")) helpers = atoi(e) - 1;
    helpers = std::max(0, std::min(helpers, 7));
    dc.copy_pool.reset(new CopyPool(helpers));
  }
  return CAPY_OK;
}

// the half must be free: its last DMA has finished and, for a device-to-host half, its bytes have been handed over
static int stage_settle(capy_ctx* ctx, DeviceCtx& dc, StageSlot& ss, int h) {
  if (!ss.pending[h]) return CAPY_OK;
  CAPY_CUDA(ctx, cudaEventSynchronize(ss.ev[h]));
  if (ss.drain_dst[h]) {
    dc.copy_pool->copy(ss.drain_dst[h], ss.p + (size_t)h * kStagePiece, ss.drain_bytes[h]);
    ss.drain_dst[h] = nullptr;
  }
  ss.pending[h] = false;
  return CAPY_OK;
}

int copy_in(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, Slot slot, void* d_dst, const void* h_src, size_t bytes) {
  if (bytes == 0) return CAPY_OK;
  if (bytes < kStageMinBytes || !host_is_pageable(h_src)) {
    CAPY_CUDA(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, st));
    return CAPY_OK;
  }
  StageSlot& ss = dc.stage[stream_set(dc, st)][slot];
  int rc = stage_ready(ctx, dc, ss);
  if (rc) return rc;
  for (size_t at = 0; at < bytes; at += kStagePiece) {
    const size_t len = std::min(kStagePiece, bytes - at);
    const int h = ss.next;
    ss.next ^= 1;
    rc = stage_settle(ctx, dc, ss, h);
    if (rc) return rc;
    uint8_t* half = ss.p + (size_t)h * kStagePiece;
    dc.copy_pool->copy(half, (const uint8_t*)h_src + at, len);
    CAPY_CUDA(ctx, cudaMemcpyAsync((uint8_t*)d_dst + at, half, len, cudaMemcpyHostToDevice, st));
    CAPY_CUDA(ctx, cudaEventRecord(ss.ev[h], st));
    ss.pending[h] = true;
  }
  return CAPY_OK;
}

int copy_out(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, Slot slot, void* h_dst, const void* d_src, size_t bytes) {
  if (bytes == 0) return CAPY_OK;
  if (bytes < kStageMinBytes || !host_is_pageable(h_dst)) {
    CAPY_CUDA(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st));
    return CAPY_OK;
  }
  StageSlot& ss = dc.stage[stream_set(dc, st)][slot];
  int rc = stage_ready(ctx, dc, ss);
  if (rc) return rc;
  for (size_t at = 0; at < bytes; at += kStagePiece) {
    const size_t len = std::min(kStagePiece, bytes - at);
    const int h = ss.next;
    ss.next ^= 1;
    rc = stage_settle(ctx, dc, ss, h);
    if (rc) return rc;
    uint8_t* half = ss.p + (size_t)h * kStagePiece;
    CAPY_CUDA(ctx, cudaMemcpyAsync(half, (const uint8_t*)d_src + at, len, cudaMemcpyDeviceToHost, st));
    CAPY_CUDA(ctx, cudaEventRecord(ss.ev[h], st));
    ss.pending[h] = true;
    ss.drain_dst[h] = (uint8_t*)h_dst + at;
    ss.drain_bytes[h] = len;
  }
  return CAPY_OK;
}

int stage_drain(capy_ctx* ctx, DeviceCtx& dc) {
  int rc = CAPY_OK;
  for (auto& set : dc.stage)
    for (StageSlot& ss : set)
      for (int h = 0; h < 2; h++)
        if (ss.pending[h]) {
          const int r = stage_settle(ctx, dc, ss, h);
          if (r && !rc) rc = r;
        }
  return rc;
}

void stage_free(DeviceCtx& dc) {
  for (auto& set : dc.stage)
    for (StageSlot& ss : set) {
      for (int h = 0; h < 2; h++)
        if (ss.ev[h]) cudaEventDestroy(ss.ev[h]);
      if (ss.p) cudaFreeHost(ss.p);
      ss = StageSlot();
    }
  dc.copy_pool.reset();
}

void plan_cache_clear(DeviceCtx& dc) {
  for (PlanEntry& e : dc.plans)
    if (e.owned_order) cudaFree(e.owned_order);  // cudaFree waits for work that still reads it
  dc.plans.clear();
}

}  // namespace capy

using namespace capy;

extern "C" {

int capy_version(void) { return 100; }

const char* capy_strerror(int status) {
  switch (status) {
    case CAPY_OK: return "ok";
    case CAPY_ERR_BAD_SECPARAM: return "unsupported security parameter (expected 224, 256, 384 or 512)";
    case CAPY_ERR_BAD_ARG: return "bad argument";
    case CAPY_ERR_CUDA: return "CUDA error (see capy_last_cuda_error)";
    case CAPY_ERR_BAD_POINT: return "input point is not on the curve";
    case CAPY_ERR_NO_DEVICE: return "no usable CUDA device";
    case CAPY_ERR_OOM: return "out of device memory";
    default: return "unknown status";
  }
}

int capy_gpu_init(const int* devices, int n_devices, capy_ctx** out_ctx) {
  if (!out_ctx) return CAPY_ERR_BAD_ARG;
  *out_ctx = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
    cudaGetLastError();
    return CAPY_ERR_NO_DEVICE;
  }
  std::vector<int> devs;
  if (!devices || n_devices <= 0) {
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) return CAPY_ERR_NO_DEVICE;
    devs.push_back(cur);
  } else {
    for (int i = 0; i < n_devices; i++) {
      if (devices[i] < 0 || devices[i] >= count) return CAPY_ERR_BAD_ARG;
      devs.push_back(devices[i]);
    }
  }
  capy_ctx* ctx = new (std::nothrow) capy_ctx();
  if (!ctx) return CAPY_ERR_OOM;
  ctx->devs.resize(devs.size());
  for (size_t i = 0; i < devs.size(); i++) {
    DeviceCtx& dc = ctx->devs[i];
    dc.dev = devs[i];
    dc.index = (int)i;
    DeviceGuard g(dc.dev);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dc.dev) != cudaSuccess) {
      capy_gpu_destroy(ctx);
      return CAPY_ERR_NO_DEVICE;
    }
    dc.sm_count = prop.multiProcessorCount;
    for (int s = 0; s < kNumStreams; s++) {
      if (cudaStreamCreateWithFlags(&dc.streams[s], cudaStreamNonBlocking) != cudaSuccess) {
        capy_gpu_destroy(ctx);
        return CAPY_ERR_CUDA;
      }
    }
  }
  if (devs.size() > 1)
    for (DeviceCtx& dc : ctx->devs) dc.worker.reset(new DeviceWorker(dc.dev));
  *out_ctx = ctx;
  return CAPY_OK;
}

void capy_gpu_destroy(capy_ctx* ctx) {
  if (!ctx) return;
  for (DeviceCtx& dc : ctx->devs) dc.worker.reset();  // joins the worker threads
  for (DeviceCtx& dc : ctx->devs) {
    DeviceGuard g(dc.dev);
    cudaDeviceSynchronize();
    plan_cache_clear(dc);
    for (int s = 0; s < kNumStreams; s++)
      if (dc.streams[s]) cudaStreamDestroy(dc.streams[s]);
    for (auto& set : dc.scratch)
      for (Scratch& sc : set)
        if (sc.p) cudaFree(sc.p);
    if (dc.vb_slabs.p) cudaFree(dc.vb_slabs.p);
    for (auto& kv : dc.prefix_cache) {
      if (kv.second.d_state) cudaFree(kv.second.d_state);
      if (kv.second.d_prefix) cudaFree(kv.second.d_prefix);
    }
    ed448_tables_free(dc);
    stage_free(dc);
  }
  delete ctx;
}

int capy_gpu_scrub(capy_ctx* ctx) {
  if (!ctx) return CAPY_ERR_BAD_ARG;
  for (DeviceCtx& dc : ctx->devs) {
    std::lock_guard<std::mutex> lk(*dc.mu);
    DeviceGuard g(dc.dev);
    CAPY_CUDA(ctx, cudaDeviceSynchronize());
    for (auto& set : dc.scratch)
      for (Scratch& sc : set)
        if (sc.p) CAPY_CUDA(ctx, cudaMemset(sc.p, 0, sc.cap));
    if (dc.vb_slabs.p) CAPY_CUDA(ctx, cudaMemset(dc.vb_slabs.p, 0, dc.vb_slabs.cap));
    CAPY_CUDA(ctx, cudaDeviceSynchronize());
    for (auto& set : dc.stage)  // the page-locked staging halves saw passwords and plaintexts too
      for (StageSlot& ss : set)
        if (ss.p) memset(ss.p, 0, 2 * kStagePiece);
  }
  return CAPY_OK;
}

int capy_gpu_set_plan_cache(capy_ctx* ctx, int enable) {
  if (!ctx) return CAPY_ERR_BAD_ARG;
  ctx->plan_cache.store(enable ? 1 : 0);
  if (!enable)
    for (DeviceCtx& dc : ctx->devs) {
      std::lock_guard<std::mutex> lk(*dc.mu);
      DeviceGuard g(dc.dev);
      plan_cache_clear(dc);
    }
  return CAPY_OK;
}

int capy_gpu_device_count(const capy_ctx* ctx) { return ctx ? (int)ctx->devs.size() : 0; }

const char* capy_last_cuda_error(const capy_ctx* ctx) { return ctx ? ctx->last_cuda_error.c_str() : ""; }

uint64_t capy_launch_count(const capy_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }

void* capy_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void capy_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

int capy_copy_probe(capy_ctx* ctx, int dev_index, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes, int reps,
                    double* ms_per_rep) {
  if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size() || !ms_per_rep || reps < 1 || (in_bytes && !h_in) ||
      (out_bytes && !h_out))
    return CAPY_ERR_BAD_ARG;
  DeviceCtx& dc = ctx->devs[dev_index];
  std::lock_guard<std::mutex> lk(*dc.mu);
  DeviceGuard g(dc.dev);
  // own buffers (not the scratch slots of the pipelines): plain copies, nothing else on the device
  void *d_in = nullptr, *d_out = nullptr;
  CAPY_CUDA(ctx, cudaMalloc(&d_in, in_bytes ? in_bytes : 16));
  if (cudaMalloc(&d_out, out_bytes ? out_bytes : 16) != cudaSuccess) {
    cudaFree(d_in);
    return cuda_fail(ctx, cudaGetLastError(), "cudaMalloc(d_out)");
  }
  cudaEvent_t e0, e1, e2;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  cudaEventCreate(&e2);
  cudaStream_t s0 = dc.streams[0], s1 = dc.streams[1];
  int rc = CAPY_OK;
  float ms = 0.f;
  for (int pass = 0; pass < 2 && rc == CAPY_OK; pass++) {  // pass 0 = warm-up
    const int n = pass == 0 ? 1 : reps;
    cudaEventRecord(e0, s0);
    cudaStreamWaitEvent(s1, e0, 0);
    for (int r = 0; r < n; r++) {
      if (in_bytes && cudaMemcpyAsync(d_in, h_in, in_bytes, cudaMemcpyHostToDevice, s0) != cudaSuccess) rc = CAPY_ERR_CUDA;
      if (out_bytes && cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, s1) != cudaSuccess) rc = CAPY_ERR_CUDA;
    }
    cudaEventRecord(e1, s1);
    cudaStreamWaitEvent(s0, e1, 0);
    cudaEventRecord(e2, s0);
    if (cudaEventSynchronize(e2) != cudaSuccess) rc = CAPY_ERR_CUDA;
    if (rc == CAPY_OK) cudaEventElapsedTime(&ms, e0, e2);
  }
  if (rc != CAPY_OK) cuda_fail(ctx, cudaGetLastError(), "capy_copy_probe");
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaEventDestroy(e2);
  cudaFree(d_in);
  cudaFree(d_out);
  *ms_per_rep = (double)ms / reps;
  return rc;
}

}  // extern "C"
