// ed448_var.cu -- variable-base scalar multiplication [k]P (ecc/signable.rs:77 `*pub_key * h_scalar`,
// ecc/encryptable.rs:37,78): signed radix-16 fixed window, per-item table 1P..8P (ed448.cuh `pt_var_base_mul`).
//
// One 256-thread block per SM, one item per thread, two warps per scheduler (measured with csrc/fe_mul_probe.cu: one warp
// alone reaches 73 % of the IMAD.WIDE issue rate, two reach it).  The table of an item (8 cached points, each packed into
// 14 uint4 chunks = 1 792 B) is thread-interleaved, 128 items to a slab:
//     slab[(entry * 14 + chunk) * 128 + thread]            8 * 14 * 128 * 16 B = 229 376 B
// so a warp reads 32 consecutive 16-byte chunks whichever entry each thread wants, and a thread only ever touches its own
// column (no barrier needed for the table).  Warps 0-3 keep their slab in SHARED memory (229 376 of the 232 448 bytes a
// block may have, which also pins the kernel to one block per SM); warps 4-7 keep theirs in a per-SM slab of global memory
// (148 x 224 KB = 34 MB for the whole GPU, indexed by %smid, reused by every block that runs on the SM: it never leaves
// the L2).  The previous version kept the table (2 KB per thread) in local memory: 98 GB of DRAM traffic per 2^18-item
// launch.
// The constant-time scan of the table is software-pipelined over half entries, so the L2 latency of the second four warps
// is covered by the masking of the previous half.  The block barrier that kept the eight warps on one instruction stream
// while the table was in local memory is gone: it cost 6 % once the table had moved (31.8 -> 29.5 ms per 2^18 items).
#ifndef CAPY_ED_MINBLOCKS
#define CAPY_ED_MINBLOCKS 1
#endif
#include "ed448_kernels.h"

namespace capy {

constexpr int VB_BLOCK = 256;  // threads per block (= per SM)
constexpr int VB_SLAB = 128;   // items per table slab
constexpr size_t VB_SLAB_BYTES = (size_t)VB_ENTRIES * VB_CHUNKS * VB_SLAB * sizeof(uint4);
constexpr size_t VB_SMEM = VB_SLAB_BYTES;

// r_i = [k_i]P_i (+ addend_i).  scalars: 56-byte big-endian, exact integers (mode4 = 0) or
// 4 * BE mod r (mode4 = 1, ECDH: ecc/encryptable.rs:36).  Off-curve P_i -> bad[i] = 1, identity out.
__global__ void __launch_bounds__(VB_BLOCK, 1) var_base_kernel(const uint8_t* __restrict__ scalars_be56, int mode4,
                                                               const uint8_t* __restrict__ points_xy,
                                                               const uint32_t* __restrict__ addend /* ext SoA or null */,
                                                               uint32_t* __restrict__ proj, uint8_t* __restrict__ bad,
                                                               uint64_t n, int constant_time, uint4* __restrict__ sm_slabs) {
  extern __shared__ uint4 vb_tab[];
  uint32_t smid;
  asm("mov.u32 %0, %%smid;" : "=r"(smid));
  // this thread's table column: shared memory for the first four warps, this SM's global slab for the other four
  uint4* col = threadIdx.x < VB_SLAB ? vb_tab + threadIdx.x
                                     : sm_slabs + (size_t)smid * (VB_SLAB_BYTES / sizeof(uint4)) + (threadIdx.x - VB_SLAB);
  // no early exits: idle threads of the last block shadow the last item and off-curve inputs run the (complete)
  // arithmetic on the identity, so every thread reaches the block barriers of the ladder
  const uint64_t gi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = gi < n;
  const uint64_t i = active ? gi : n - 1;
  Sc k;
  sc_from_be(k, scalars_be56 + 56 * i);
  if (mode4) {
    Sc t = k;
    sc_mul4_mod(k, t);
  }
  PtExt r;
  bool ok;
  {
    uint32_t w[14];
    Fe x, y;
    const uint8_t* pb = points_xy + 112 * i;
#pragma unroll
    for (int j = 0; j < 14; j++) w[j] = (uint32_t)pb[4 * j] | ((uint32_t)pb[4 * j + 1] << 8) | ((uint32_t)pb[4 * j + 2] << 16) | ((uint32_t)pb[4 * j + 3] << 24);
    fe_from_words(x, w);
#pragma unroll
    for (int j = 0; j < 14; j++) w[j] = (uint32_t)pb[56 + 4 * j] | ((uint32_t)pb[57 + 4 * j] << 8) | ((uint32_t)pb[58 + 4 * j] << 16) | ((uint32_t)pb[59 + 4 * j] << 24);
    fe_from_words(y, w);
    ok = pt_from_affine(r, x, y);
    if (!ok) pt_identity(r);
  }
  pt_var_base_mul<VB_SLAB>(r, k, col, constant_time != 0, addend != nullptr, [&](PtExt& a) {
#pragma unroll
    for (int j = 0; j < 16; j++) {
      a.X.v[j] = addend[(uint64_t)(j)*n + i];
      a.Y.v[j] = addend[(uint64_t)(16 + j) * n + i];
      a.Z.v[j] = addend[(uint64_t)(32 + j) * n + i];
      a.T.v[j] = addend[(uint64_t)(48 + j) * n + i];
    }
  });
  if (!ok) pt_identity(r);  // off-curve input: identity out, no addend (the caller reports the item as bad)
  if (active) {
    if (bad) bad[i] = ok ? 0 : 1;
    store_ext(proj, n, i, r);
  }
}

int launch_var_base(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint8_t* scalars, int mode4, const uint8_t* points,
                    const uint32_t* addend, uint32_t* proj, uint8_t* bad, uint64_t n, bool constant_time) {
  // per-SM table slabs of the second half of every block (a fixed 34 MB per device, allocated once)
  uint4* slabs = (uint4*)scratch_grow(dc.vb_slabs, (size_t)dc.sm_count * VB_SLAB_BYTES);
  if (!slabs) return CAPY_ERR_OOM;
  CAPY_CUDA(ctx, cudaFuncSetAttribute(var_base_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VB_SMEM));
  var_base_kernel<<<grid_for(n, VB_BLOCK), VB_BLOCK, VB_SMEM, st>>>(scalars, mode4, points, addend, proj, bad, n,
                                                                     constant_time ? 1 : 0, slabs);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

}  // namespace capy
