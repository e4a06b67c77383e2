// ed448_fixed.cu -- fixed-base scalar multiplication [k]G: comb table of G built once per device,
// then 112 mixed additions per item (the reference has no fixed-base path: `generator() * s` runs the
// generic Mul<Scalar>, ecc/keypair.rs:44; the result is the same curve point).
#ifndef CAPY_ED_MINBLOCKS
#define CAPY_ED_MINBLOCKS 1
#endif
#include "ed448_kernels.h"

namespace capy {

struct Ed448Tables {
  uint32_t* fb = nullptr;  // [112][8][48] comb table of G
};

void ed448_tables_free(DeviceCtx& dc) {
  if (dc.ed) {
    if (dc.ed->fb) cudaFree(dc.ed->fb);
    delete dc.ed;
    dc.ed = nullptr;
  }
}

// points_xy == nullptr: thread i builds window i of G's table.  Otherwise thread t converts the affine point t of
// points_xy (112 bytes: x || y), the multiple (j+1) * 32^i * V with t = 16 i + j, into entry t of V's table.
__global__ void fb_table_kernel(uint32_t* table, const uint8_t* __restrict__ points_xy) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (!points_xy) {
    if (t < FB_WINDOWS) fb_build_window(table + (size_t)t * FB_ENTRIES * FB_ENTRY_WORDS, t);
    return;
  }
  if (t < FB_WINDOWS * FB_ENTRIES) fb_niels_entry_xy(table + (size_t)t * FB_ENTRY_WORDS, points_xy + 112 * (size_t)t);
}

// r_i = [k_i]G, k_i reduced scalars in SoA words; result stored extended (X, Y, Z, T).  `table` is the comb table of
// phi(G) or of another point of order r.  With table2 the kernel runs a second pass of FB_WINDOWS windows over the
// digits of k2_i and table2 into the same accumulator: r_i = [k_i]G + [k2_i]V (G and V of odd order r, so the dual
// isogeny of the sum is exact).
// All threads of a block walk the windows in lock step, so the 3 KB table row of window w+1 is copied to
// shared memory with cp.async while window w is being added (double buffer, one barrier per window); the
// constant-time scan then reads broadcast shared-memory words instead of waiting on L1/L2.
__global__ void __launch_bounds__(128, CAPY_ED_MINBLOCKS) fixed_base_kernel(const uint32_t* __restrict__ k_words,
                                                                            const uint32_t* __restrict__ table,
                                                                            uint32_t* __restrict__ proj, uint64_t n,
                                                                            int constant_time,
                                                                            const uint32_t* __restrict__ k2_words,
                                                                            const uint32_t* __restrict__ table2) {
  constexpr int ROW_WORDS = FB_ENTRIES * FB_ENTRY_WORDS;  // 768 words = 192 x 16 B
  __shared__ __align__(16) uint32_t rows[2][ROW_WORDS];
  const uint64_t gi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = gi < n;
  const uint64_t i = active ? gi : n - 1;  // idle threads of the last block shadow the last item (barriers)
  const int windows = table2 ? 2 * FB_WINDOWS : FB_WINDOWS;
  auto stage = [&](int buf, int win) {  // win counts the windows of both passes
    const uint32_t* src = win < FB_WINDOWS ? table + (size_t)win * ROW_WORDS : table2 + (size_t)(win - FB_WINDOWS) * ROW_WORDS;
    for (int c = threadIdx.x; c < ROW_WORDS / 4; c += blockDim.x) {
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&rows[buf][4 * c]);
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src + 4 * c));
    }
    asm volatile("cp.async.commit_group;");
  };
  stage(0, 0);
  PtExt acc;
  pt_identity(acc);
#pragma unroll 1
  for (int w0 = 0; w0 < windows; w0 += FB_WINDOWS) {
    const uint32_t* kw = w0 ? k2_words : k_words;
    Sc k, kq;
#pragma unroll
    for (int j = 0; j < 14; j++) k.w[j] = kw[(uint64_t)j * n + i];
    const Sc inv4 = {CAPY_INV4_LIMBS};
    sc_mul_mod(kq, k, inv4);  // k / 4 mod r: the comb runs on the 4-isogenous curve
    uint32_t carry = 0;       // ends at 0: kq < 2^446
#pragma unroll 1
    for (int w = w0; w < w0 + FB_WINDOWS; w++) {
      asm volatile("cp.async.wait_group 0;");
      __syncthreads();  // row w is visible to everyone; everyone has finished reading row w - 1
      if (w + 1 < windows) stage((w + 1) & 1, w + 1);
      const int dgt = fb_digit(kq, w - w0, carry);
      PtNiels e;
      fb_lookup_row<true>(e, rows[w & 1], dgt, constant_time != 0);
      pt_madd_tw<true>(acc, acc, e);
    }
  }
  PtExt r;
  pt_dual_isogeny(r, acc);
  if (active) store_ext(proj, n, i, r);
}

static int ensure_tables(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t stream) {
  if (dc.ed && dc.ed->fb) return CAPY_OK;
  if (!dc.ed) dc.ed = new Ed448Tables();
  const size_t bytes = (size_t)FB_WINDOWS * FB_ENTRIES * FB_ENTRY_WORDS * sizeof(uint32_t);
  uint32_t* fb = nullptr;
  CAPY_CUDA(ctx, cudaMalloc(&fb, bytes));
  dc.ed->fb = fb;
  fb_table_kernel<<<(FB_WINDOWS + 31) / 32, 32, 0, stream>>>(dc.ed->fb, nullptr);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  // once per device: later calls may launch on other (non-blocking) streams and must not see a half-built table
  CAPY_CUDA(ctx, cudaStreamSynchronize(stream));
  return CAPY_OK;
}

int launch_fixed_base(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint32_t* k_words, uint32_t* proj, uint64_t n,
                      bool constant_time, const uint32_t* table, const uint32_t* k2_words, const uint32_t* table2) {
  if (!table) {
    int rc = ensure_tables(ctx, dc, st);
    if (rc) return rc;
    table = dc.ed->fb;
  }
  fixed_base_kernel<<<grid_for(n, 128), 128, 0, st>>>(k_words, table, proj, n, constant_time ? 1 : 0, k2_words, table2);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

int launch_fb_table_from_points(capy_ctx* ctx, cudaStream_t st, const uint8_t* points_xy, uint32_t* table) {
  fb_table_kernel<<<grid_for(FB_WINDOWS * FB_ENTRIES, 128), 128, 0, st>>>(table, points_xy);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

}  // namespace capy
