// ed448_kernels.h -- launchers shared by the Ed448 translation units (split so they compile in parallel).
#pragma once
#include "ed448.cuh"
#include "internal.h"

namespace capy {

// extended point of item i, limb-major SoA: word w at proj[w * n + i], w = 0..63 (X | Y | Z | T)
__device__ __forceinline__ void store_ext(uint32_t* __restrict__ proj, uint64_t n, uint64_t i, const PtExt& p) {
#pragma unroll
  for (int k = 0; k < 16; k++) {
    proj[(uint64_t)(k)*n + i] = p.X.v[k];
    proj[(uint64_t)(16 + k) * n + i] = p.Y.v[k];
    proj[(uint64_t)(32 + k) * n + i] = p.Z.v[k];
    proj[(uint64_t)(48 + k) * n + i] = p.T.v[k];
  }
}

// ed448_fixed.cu
// proj = [k]G, or [k]V with `table` = the comb table of V; with table2 also + [k2]V2 (joint comb, one launch)
int launch_fixed_base(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint32_t* k_words, uint32_t* proj, uint64_t n,
                      bool constant_time, const uint32_t* table = nullptr, const uint32_t* k2_words = nullptr,
                      const uint32_t* table2 = nullptr);
// table := comb table of V from the FB_WINDOWS * FB_ENTRIES affine multiples (j+1) * 32^i * V, item 16 i + j
int launch_fb_table_from_points(capy_ctx* ctx, cudaStream_t st, const uint8_t* points_xy, uint32_t* table);
constexpr size_t kFbTableBytes = (size_t)FB_WINDOWS * FB_ENTRIES * FB_ENTRY_WORDS * sizeof(uint32_t);
// ed448_var.cu
int launch_var_base(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint8_t* scalars, int mode4, const uint8_t* points,
                    const uint32_t* addend, uint32_t* proj, uint8_t* bad, uint64_t n, bool constant_time);

// ed448_api.cu
int launch_scalar_prep(capy_ctx* ctx, cudaStream_t st, const uint8_t* in, int mode, uint32_t* words, uint8_t* be, uint64_t n);
int launch_to_affine(capy_ctx* ctx, cudaStream_t st, const uint32_t* proj, uint64_t n, int mode, const uint8_t* bad, uint8_t* out);
// *bad_flag |= 1 when any of bad[0 .. n) is set
int launch_any_bad(capy_ctx* ctx, cudaStream_t st, const uint8_t* bad, int* bad_flag, uint64_t n);
// out[0 .. n) := the 112 bytes at d_xy (device to device copies)
int broadcast_point(capy_ctx* ctx, cudaStream_t st, const uint8_t* d_xy, uint8_t* out, uint64_t n);
// CAPY_ERR_BAD_ARG unless key was prepared by ctx
int pub_check(const capy_ctx* ctx, const capy_ed448_pub* key);
int dev_secret_scalar(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* d_pws, const uint64_t* d_pw_off,
                      uint64_t n, uint32_t* s_words, uint8_t* s_be);

}  // namespace capy
