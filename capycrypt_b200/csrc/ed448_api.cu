// ed448_api.cu -- Ed448 batch entry points (C ABI in include/capy_gpu.h).
//
// Replaces, for batches, KeyPair::new (ecc/keypair.rs:41-51), Signable::sign / verify
// (ecc/signable.rs:40-57, 72-86) and the scalar-multiplication core of KeyEncryptable
// (ecc/encryptable.rs:36-38, 76-78).  A pipeline is a short chain of kernels on one stream:
// KMACXOF (sponge kernel) -> scalar glue (mod r) -> scalar multiplication -> batched inversion
// to affine -> KMACXOF ... .  Keccak (72 registers) and the curve kernels (~250 registers) are
// deliberately separate launches; intermediate points live in HBM in limb-major SoA layout
// (word w of item i at [w * n + i]) so that every access is coalesced.
#include <cstring>

#include "ed448_kernels.h"
#include "hostbatch.h"

namespace capy {

// scalar glue.  in: 56-byte big-endian integers.  mode 0: o = in mod r ; mode 1: o = 4 * in mod r
// (bytes_to_scalar(..).mul_mod(&Scalar::from(4)), ecc/keypair.rs:43).  Writes the scalar as 14
// words (SoA) and optionally as 56 bytes big-endian (scalar_to_bytes, the "N" KMAC key in sign).
__global__ void __launch_bounds__(128) scalar_prep_kernel(const uint8_t* __restrict__ in_be56, int mode,
                                                          uint32_t* __restrict__ out_words, uint8_t* __restrict__ out_be56,
                                                          uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Sc a, o;
  sc_from_be(a, in_be56 + 56 * i);
  if (mode == 1) sc_mul4_mod(o, a);
  else sc_reduce_448(o, a);
#pragma unroll
  for (int k = 0; k < 14; k++) out_words[(uint64_t)k * n + i] = o.w[k];
  if (out_be56) sc_to_be(out_be56 + 56 * i, o);
}

// z = k - (BE(h) * s mod r) mod r   (ecc/signable.rs:52-54)
__global__ void __launch_bounds__(128) sign_finish_kernel(const uint32_t* __restrict__ k_words,
                                                          const uint32_t* __restrict__ s_words,
                                                          const uint8_t* __restrict__ h56, uint8_t* __restrict__ z_be56,
                                                          uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Sc k, s, h, hs, z;
#pragma unroll
  for (int j = 0; j < 14; j++) {
    k.w[j] = k_words[(uint64_t)j * n + i];
    s.w[j] = s_words[(uint64_t)j * n + i];
  }
  sc_from_be(h, h56 + 56 * i);
  sc_mul_mod(hs, h, s);
  sc_sub_mod(z, k, hs);
  sc_to_be(z_be56 + 56 * i, z);
}

// to_affine for a whole batch with Montgomery's trick: each thread inverts the product of K
// Z-coordinates (items t, t + T, t + 2T, ...: coalesced) and unwinds it, so an item costs ~5 field
// multiplications plus 1/K of an inversion instead of a full inversion (FieldElement inversion in
// ExtendedPoint::to_affine, ecc/signable.rs:49,79).  mode 0: x || y (112 B); mode 1: x only (56 B).
template <int K>
__global__ void __launch_bounds__(128) to_affine_kernel(const uint32_t* __restrict__ proj, uint64_t n, int mode,
                                                        const uint8_t* __restrict__ bad, uint8_t* __restrict__ out) {
  const uint64_t T = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  Fe pre[K];  // pre[j] = Z_0 * ... * Z_j
  int cnt = 0;
#pragma unroll 1
  for (int j = 0; j < K; j++) {
    const uint64_t i = t + (uint64_t)j * T;
    if (i >= n) break;
    Fe z;
#pragma unroll
    for (int k = 0; k < 16; k++) z.v[k] = proj[(uint64_t)(32 + k) * n + i];
    if (j == 0) fe_copy(pre[0], z);
    else fe_mul(pre[j], pre[j - 1], z);
    cnt++;
  }
  Fe inv;
  fe_inv(inv, pre[cnt - 1]);
  const uint32_t out_stride = mode == 0 ? 112u : 56u;
#pragma unroll 1
  for (int j = cnt - 1; j >= 0; j--) {
    const uint64_t i = t + (uint64_t)j * T;
    Fe zi, z, x, y;
    if (j > 0) {
      fe_mul(zi, inv, pre[j - 1]);
#pragma unroll
      for (int k = 0; k < 16; k++) z.v[k] = proj[(uint64_t)(32 + k) * n + i];
      fe_mul(inv, inv, z);
    } else {
      fe_copy(zi, inv);
    }
#pragma unroll
    for (int k = 0; k < 16; k++) x.v[k] = proj[(uint64_t)k * n + i];
    fe_mul(x, x, zi);
    uint32_t w[14];
    fe_to_words(w, x);
    const bool zero_it = bad && bad[i];
    uint8_t* o = out + (uint64_t)out_stride * i;
    // 56- and 112-byte rows are 8-byte aligned when the base is
    if ((reinterpret_cast<uintptr_t>(out) & 7u) == 0) {
#pragma unroll
      for (int k = 0; k < 7; k++) reinterpret_cast<uint2*>(o)[k] = zero_it ? make_uint2(0, 0) : make_uint2(w[2 * k], w[2 * k + 1]);
    } else {
      for (int k = 0; k < 56; k++) o[k] = zero_it ? 0 : (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
    }
    if (mode == 0) {
#pragma unroll
      for (int k = 0; k < 16; k++) y.v[k] = proj[(uint64_t)(16 + k) * n + i];
      fe_mul(y, y, zi);
      fe_to_words(w, y);
      if ((reinterpret_cast<uintptr_t>(out) & 7u) == 0) {
#pragma unroll
        for (int k = 0; k < 7; k++) reinterpret_cast<uint2*>(o + 56)[k] = zero_it ? make_uint2(0, 0) : make_uint2(w[2 * k], w[2 * k + 1]);
      } else {
        for (int k = 0; k < 56; k++) o[56 + k] = zero_it ? 0 : (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
      }
    }
  }
}

// ok[i] = (h'_i == h_i) && !bad[i]   (ecc/signable.rs:81-85)
__global__ void verify_compare_kernel(const uint8_t* __restrict__ hp, const uint8_t* __restrict__ h,
                                      const uint8_t* __restrict__ bad, uint8_t* __restrict__ ok, int* bad_flag, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t diff = 0;
  for (int k = 0; k < 56; k++) diff |= (uint32_t)(hp[56 * i + k] ^ h[56 * i + k]);
  const bool b = bad && bad[i];
  ok[i] = (diff == 0 && !b) ? 1 : 0;
  if (b && bad_flag) atomicOr(bad_flag, 1);
}

__global__ void any_bad_kernel(const uint8_t* __restrict__ bad, int* bad_flag, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && bad[i]) atomicOr(bad_flag, 1);
}

// ---- launch helpers ----------------------------------------------------------------------------------
constexpr int kInvBatch = 16;

int launch_scalar_prep(capy_ctx* ctx, cudaStream_t st, const uint8_t* in, int mode, uint32_t* words, uint8_t* be,
                              uint64_t n) {
  scalar_prep_kernel<<<grid_for(n, 128), 128, 0, st>>>(in, mode, words, be, n);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

int launch_to_affine(capy_ctx* ctx, cudaStream_t st, const uint32_t* proj, uint64_t n, int mode, const uint8_t* bad,
                            uint8_t* out) {
  const uint64_t threads = (n + kInvBatch - 1) / kInvBatch;
  to_affine_kernel<kInvBatch><<<grid_for(threads, 128), 128, 0, st>>>(proj, n, mode, bad, out);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

int launch_verify_compare(capy_ctx* ctx, cudaStream_t st, const uint8_t* hp, const uint8_t* h, const uint8_t* bad, uint8_t* ok,
                          int* bad_flag, uint64_t n) {
  verify_compare_kernel<<<grid_for(n, 256), 256, 0, st>>>(hp, h, bad, ok, bad_flag, n);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

int launch_any_bad(capy_ctx* ctx, cudaStream_t st, const uint8_t* bad, int* bad_flag, uint64_t n) {
  any_bad_kernel<<<grid_for(n, 256), 256, 0, st>>>(bad, bad_flag, n);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

// ---- device pipelines (async on `st`) ----------------------------------------------------------------
static int dev_fixed_base(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint8_t* d_scalars, uint64_t n,
                          uint8_t* d_out_xy) {
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(kw, uint32_t, kEdKWords, n * 56);
  CAPY_SCRATCH(proj, uint32_t, kEdProj, n * 256);
  int rc = launch_scalar_prep(ctx, st, d_scalars, 0, kw, nullptr, n);
  if (rc) return rc;
  rc = launch_fixed_base(ctx, dc, st, kw, proj, n, true);
  if (rc) return rc;
  return launch_to_affine(ctx, st, proj, n, 0, nullptr, d_out_xy);
}

static int dev_var_base(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint8_t* d_scalars, const uint8_t* d_points,
                        uint64_t n, uint8_t* d_out_xy, int* d_bad_flag) {
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(proj, uint32_t, kEdProj, n * 256);
  CAPY_SCRATCH(bad, uint8_t, kEdBad, n);
  int rc = launch_var_base(ctx, dc, st, d_scalars, 0, d_points, nullptr, proj, bad, n, true);
  if (rc) return rc;
  rc = launch_to_affine(ctx, st, proj, n, 0, bad, d_out_xy);
  if (rc) return rc;
  return d_bad_flag ? launch_any_bad(ctx, st, bad, d_bad_flag, n) : CAPY_OK;
}

// s = 4 * BE(KMACXOF(pw, "", 448, "SK", d)) mod r  (ecc/keypair.rs:42-43): words + optional BE bytes
int dev_secret_scalar(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* d_pws,
                             const uint64_t* d_pw_off, uint64_t n, uint32_t* s_words, uint8_t* s_be) {
  CAPY_SCRATCH(tmp, uint8_t, kEdTmp56A, n * 56);
  KmacPass a(d, "SK", n);
  a.job.keys = d_pws;
  a.job.key_off = d_pw_off;
  a.job.out_bytes = a.job.out_stride = 56;  // 448 bits
  a.job.out = tmp;
  int rc = launch_kmac_xof(ctx, dc, st, a);
  if (rc) return rc;
  return launch_scalar_prep(ctx, st, tmp, 1, s_words, s_be, n);
}

static int dev_keygen(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* d_pws, const uint64_t* d_pw_off,
                      uint64_t n, uint8_t* d_out_xy) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(sw, uint32_t, kEdSWords, n * 56);
  CAPY_SCRATCH(proj, uint32_t, kEdProj, n * 256);
  int rc = dev_secret_scalar(ctx, dc, st, d, d_pws, d_pw_off, n, sw, nullptr);
  if (rc) return rc;
  rc = launch_fixed_base(ctx, dc, st, sw, proj, n, true);
  if (rc) return rc;
  return launch_to_affine(ctx, st, proj, n, 0, nullptr, d_out_xy);
}

static int dev_sign(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* d_pws, const uint64_t* d_pw_off,
                    const uint8_t* d_msgs, const uint64_t* d_msg_off, uint64_t n, uint8_t* d_h, uint8_t* d_z) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(sw, uint32_t, kEdSWords, n * 56);
  CAPY_SCRATCH(kw, uint32_t, kEdKWords, n * 56);
  CAPY_SCRATCH(proj, uint32_t, kEdProj, n * 256);
  CAPY_SCRATCH(s_be, uint8_t, kEdTmp56B, n * 56);
  CAPY_SCRATCH(tmp, uint8_t, kEdTmp56C, n * 56);
  // s (signable.rs:41-43)
  int rc = dev_secret_scalar(ctx, dc, st, d, d_pws, d_pw_off, n, sw, s_be);
  if (rc) return rc;
  // k = 4 * BE(KMACXOF(s_bytes, m, 448, "N")) mod r (:45-46)
  KmacPass k(d, "N", n);
  k.job.keys = s_be;
  k.job.key_stride = k.job.key_len = 56;
  k.job.data = d_msgs;
  k.job.off = d_msg_off;
  k.job.out_bytes = k.job.out_stride = 56;
  k.job.out = tmp;
  rc = launch_kmac_xof(ctx, dc, st, k);
  if (rc) return rc;
  rc = launch_scalar_prep(ctx, st, tmp, 1, kw, nullptr, n);
  if (rc) return rc;
  // U = [k]G ; ux = U.to_affine().x.to_bytes() (:48-49)
  rc = launch_fixed_base(ctx, dc, st, kw, proj, n, true);
  if (rc) return rc;
  rc = launch_to_affine(ctx, st, proj, n, 1, nullptr, tmp);
  if (rc) return rc;
  // h = KMACXOF(ux, m, 448, "T") (:51): the pass of k with another key, output and customisation string
  KmacPass h = k;
  h.custom = "T";
  h.job.keys = tmp;
  h.job.out = d_h;
  rc = launch_kmac_xof(ctx, dc, st, h);
  if (rc) return rc;
  // z = k - h * s mod r (:52-54)
  sign_finish_kernel<<<grid_for(n, 128), 128, 0, st>>>(kw, sw, d_h, d_z, n);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

// Where a verification stream (capy_ed448_verify_stream_new) starts: U'.x and the off-curve flags (nullptr: none), in
// scratch of the stream that computed them
struct VerifyStart {
  const uint8_t* ux = nullptr;
  const uint8_t* bad = nullptr;
};

// ux = U.x ; h' = KMACXOF(ux, m, 448, "T") ; ok = (h' == h) && !bad   (signable.rs:78-85).  With `start`, only ux: the
// rest is the verification stream's.
static int verify_finish(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint32_t* proj_u, const uint8_t* d_msgs,
                         const uint64_t* d_msg_off, const uint8_t* d_h, const uint8_t* bad, uint64_t n, uint8_t* d_ok,
                         int* d_bad_flag, VerifyStart* start = nullptr) {
  CAPY_SCRATCH(ux, uint8_t, kEdTmp56A, n * 56);
  CAPY_SCRATCH(hp, uint8_t, kEdTmp56B, n * 56);
  int rc = launch_to_affine(ctx, st, proj_u, n, 1, nullptr, ux);
  if (rc) return rc;
  if (start) {
    start->ux = ux;
    start->bad = bad;
    return CAPY_OK;
  }
  KmacPass h(d, "T", n);
  h.job.keys = ux;
  h.job.key_stride = h.job.key_len = 56;
  h.job.data = d_msgs;
  h.job.off = d_msg_off;
  h.job.out_bytes = h.job.out_stride = 56;
  h.job.out = hp;
  rc = launch_kmac_xof(ctx, dc, st, h);
  if (rc) return rc;
  verify_compare_kernel<<<grid_for(n, 256), 256, 0, st>>>(hp, d_h, bad, d_ok, d_bad_flag, n);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

static int dev_verify(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* d_pub, const uint8_t* d_msgs,
                      const uint64_t* d_msg_off, const uint8_t* d_h, const uint8_t* d_z, uint64_t n, uint8_t* d_ok,
                      int* d_bad_flag, VerifyStart* start = nullptr) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(kw, uint32_t, kEdKWords, n * 56);
  CAPY_SCRATCH(projA, uint32_t, kEdProj, n * 256);
  CAPY_SCRATCH(projB, uint32_t, kEdProj2, n * 256);
  CAPY_SCRATCH(bad, uint8_t, kEdBad, n);
  // U = [z]G + [BE(h)]V with h unreduced (signable.rs:76-77, quirk Q10).  All inputs are public:
  // table lookups are direct, not scanned.
  int rc = launch_scalar_prep(ctx, st, d_z, 0, kw, nullptr, n);
  if (rc) return rc;
  rc = launch_fixed_base(ctx, dc, st, kw, projA, n, false);
  if (rc) return rc;
  rc = launch_var_base(ctx, dc, st, d_h, 0, d_pub, projA, projB, bad, n, false);
  if (rc) return rc;
  return verify_finish(ctx, dc, st, d, projB, d_msgs, d_msg_off, d_h, bad, n, d_ok, d_bad_flag, start);
}

// W = [k]V with k = 4 * BE(rand) mod r (ecc/encryptable.rs:36-37): W.x ; optionally Z = [k]G (:38)
static int dev_ecdh(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const uint8_t* d_k, const uint8_t* d_pub, uint64_t n,
                    uint8_t* d_wx, uint8_t* d_z_xy, int* d_bad_flag) {
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(proj, uint32_t, kEdProj, n * 256);
  CAPY_SCRATCH(bad, uint8_t, kEdBad, n);
  int rc = launch_var_base(ctx, dc, st, d_k, 1, d_pub, nullptr, proj, bad, n, true);
  if (rc) return rc;
  rc = launch_to_affine(ctx, st, proj, n, 1, bad, d_wx);
  if (rc) return rc;
  if (d_bad_flag) {
    rc = launch_any_bad(ctx, st, bad, d_bad_flag, n);
    if (rc) return rc;
  }
  if (!d_z_xy) return CAPY_OK;
  CAPY_SCRATCH(kw, uint32_t, kEdKWords, n * 56);
  rc = launch_scalar_prep(ctx, st, d_k, 1, kw, nullptr, n);
  if (rc) return rc;
  rc = launch_fixed_base(ctx, dc, st, kw, proj, n, true);
  if (rc) return rc;
  return launch_to_affine(ctx, st, proj, n, 0, nullptr, d_z_xy);
}

// ---- prepared public keys ------------------------------------------------------------------------------
// out[0 .. n) := the 112 bytes at d_xy: one copy, then ceil(log2 n) copies that double what is there
int broadcast_point(capy_ctx* ctx, cudaStream_t st, const uint8_t* d_xy, uint8_t* out, uint64_t n) {
  if (n == 0) return CAPY_OK;
  CAPY_CUDA(ctx, cudaMemcpyAsync(out, d_xy, 112, cudaMemcpyDeviceToDevice, st));
  for (uint64_t have = 1; have < n; have *= 2)
    CAPY_CUDA(ctx, cudaMemcpyAsync(out + 112 * have, out, 112 * std::min(have, n - have), cudaMemcpyDeviceToDevice, st));
  return CAPY_OK;
}

// U = [z]G + [h]V for a prepared V, then as dev_verify
static int dev_verify_prepared(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const capy_ed448_pub* key,
                               const uint8_t* d_msgs, const uint64_t* d_msg_off, const uint8_t* d_h, const uint8_t* d_z,
                               uint64_t n, uint8_t* d_ok, VerifyStart* start = nullptr) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  const uint32_t* v_table = key->d_table[dc.index];
  if (!v_table) {  // V has a torsion component: the variable-base pipeline with V repeated
    CAPY_SCRATCH(pub, uint8_t, kEdPubRep, n * 112);
    const int rc = broadcast_point(ctx, st, key->d_xy[dc.index], pub, n);
    if (rc) return rc;
    return dev_verify(ctx, dc, st, d, pub, d_msgs, d_msg_off, d_h, d_z, n, d_ok, nullptr, start);
  }
  CAPY_SCRATCH(zw, uint32_t, kEdKWords, n * 56);
  CAPY_SCRATCH(hw, uint32_t, kEdSWords, n * 56);
  CAPY_SCRATCH(proj, uint32_t, kEdProj, n * 256);
  // One joint comb over G's and V's tables.  The reference multiplies V by the unreduced integer h (quirk Q10); h mod r
  // gives the same point only because V has order r, which preparation checked ([r]V = identity) before it built V's
  // table.  All inputs are public: table lookups are direct, not scanned.
  int rc = launch_scalar_prep(ctx, st, d_z, 0, zw, nullptr, n);
  if (rc) return rc;
  rc = launch_scalar_prep(ctx, st, d_h, 0, hw, nullptr, n);
  if (rc) return rc;
  rc = launch_fixed_base(ctx, dc, st, zw, proj, n, false, nullptr, hw, v_table);
  if (rc) return rc;
  return verify_finish(ctx, dc, st, d, proj, d_msgs, d_msg_off, d_h, nullptr, n, d_ok, nullptr, start);
}

int pub_check(const capy_ctx* ctx, const capy_ed448_pub* key) {
  return key && key->ctx == ctx ? CAPY_OK : CAPY_ERR_BAD_ARG;
}

// the items of the table build: (j+1) * 32^i * V for i < FB_WINDOWS, j < FB_ENTRIES (item 16 i + j), then [r]V
constexpr uint64_t kPubTableItems = (uint64_t)FB_WINDOWS * FB_ENTRIES;

static std::vector<uint8_t> pub_table_scalars() {
  std::vector<uint8_t> s((kPubTableItems + 1) * 56);
  for (int i = 0; i < FB_WINDOWS; i++) {
    Sc p = {};
    p.w[(FB_WBITS * i) >> 5] = 1u << ((FB_WBITS * i) & 31);  // 32^i < r
    for (int j = 0; j < FB_ENTRIES; j++) {
      Sc m = {}, o;
      m.w[0] = (uint32_t)(j + 1);
      sc_mul_mod(o, p, m);
      sc_to_be(&s[56 * (FB_ENTRIES * i + j)], o);
    }
  }
  const Sc r = {CAPY_R_LIMBS};
  sc_to_be(&s[56 * kPubTableItems], r);
  return s;
}

struct DevTemp {  // cudaMalloc'ed for the duration of a scope
  void* p = nullptr;
  ~DevTemp() {
    if (p) cudaFree(p);
  }
};

// V's bytes on this device and, when *comb (on entry: still possible), its comb table: the multiples through the
// variable-base pipeline (public scalars, direct lookups), to affine, into table entries (fb_table_kernel).  *comb is
// cleared when [r]V is not the identity.
static int pub_build_device(capy_ctx* ctx, DeviceCtx& dc, const std::vector<uint8_t>& scalars, capy_ed448_pub* key,
                            bool* comb) {
  const cudaStream_t st = dc.streams[0];
  const int k = dc.index;
  CAPY_CUDA(ctx, cudaMalloc(&key->d_xy[k], 112));
  CAPY_CUDA(ctx, cudaMemcpy(key->d_xy[k], key->xy, 112, cudaMemcpyHostToDevice));
  if (!*comb) return CAPY_OK;
  const uint64_t m = kPubTableItems + 1;
  DevTemp sc, pts, proj, aff;
  CAPY_CUDA(ctx, cudaMalloc(&sc.p, m * 56));
  CAPY_CUDA(ctx, cudaMalloc(&pts.p, m * 112));
  CAPY_CUDA(ctx, cudaMalloc(&proj.p, m * 256));
  CAPY_CUDA(ctx, cudaMalloc(&aff.p, m * 112));
  CAPY_CUDA(ctx, cudaMemcpyAsync(sc.p, scalars.data(), m * 56, cudaMemcpyHostToDevice, st));
  int rc = broadcast_point(ctx, st, key->d_xy[k], (uint8_t*)pts.p, m);
  if (rc) return rc;
  rc = launch_var_base(ctx, dc, st, (const uint8_t*)sc.p, 0, (const uint8_t*)pts.p, nullptr, (uint32_t*)proj.p, nullptr, m,
                       false);
  if (rc) return rc;
  rc = launch_to_affine(ctx, st, (const uint32_t*)proj.p, m, 0, nullptr, (uint8_t*)aff.p);
  if (rc) return rc;
  uint8_t rv[112];
  CAPY_CUDA(ctx, cudaMemcpyAsync(rv, (const uint8_t*)aff.p + 112 * kPubTableItems, 112, cudaMemcpyDeviceToHost, st));
  CAPY_CUDA(ctx, cudaStreamSynchronize(st));
  bool identity = rv[56] == 1;  // (0, 1)
  for (int b = 0; b < 112; b++)
    if (b != 56 && rv[b]) identity = false;
  if (!identity) {
    *comb = false;
    return CAPY_OK;
  }
  CAPY_CUDA(ctx, cudaMalloc(&key->d_table[k], kFbTableBytes));
  rc = launch_fb_table_from_points(ctx, st, (const uint8_t*)aff.p, key->d_table[k]);
  if (rc) return rc;
  // later calls may launch on other (non-blocking) streams and must not see a half-built table
  CAPY_CUDA(ctx, cudaStreamSynchronize(st));
  return CAPY_OK;
}

// ---- host wrappers -------------------------------------------------------------------------------------
// The chunks of one device's shard (run_chunks).  At least 2^18 items: the pipelines contain latency-bound steps (the
// batch inversion of to_affine_kernel runs 16 items per thread, ~0.3 ms however few) that smaller chunks would repeat too
// often -- measured: four chunks of 2^16 through capy_ed448_fixed_base_batch 7.05 ms against 6.9 ms unchunked, although
// the copies (0.8 ms) were hidden.
static std::vector<Range> ed_chunks(Range sh) {
  const uint64_t items = sh.i1 - sh.i0;
  const size_t count = items < (1ull << 19) ? 1 : (size_t)std::min<uint64_t>(8, items >> 18);
  return split_items(nullptr, 1, sh.i0, sh.i1, count, 0);
}

}  // namespace capy

using namespace capy;

extern "C" {

int capy_ed448_fixed_base_batch_dev(capy_ctx* ctx, int dev_index, void* stream, const uint8_t* d_scalars_be56, uint64_t n,
                                    uint8_t* d_out_xy112) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_scalars_be56 || !d_out_xy112)) return CAPY_ERR_BAD_ARG;
  return dev_fixed_base(ctx, dc, st, d_scalars_be56, n, d_out_xy112);
}

int capy_ed448_var_base_batch_dev(capy_ctx* ctx, int dev_index, void* stream, const uint8_t* d_scalars_be56,
                                  const uint8_t* d_points_xy112, uint64_t n, uint8_t* d_out_xy112, int* d_bad_flag) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_scalars_be56 || !d_points_xy112 || !d_out_xy112)) return CAPY_ERR_BAD_ARG;
  return dev_var_base(ctx, dc, st, d_scalars_be56, d_points_xy112, n, d_out_xy112, d_bad_flag);
}

int capy_ed448_keygen_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pws,
                                const uint64_t* d_pw_off, uint64_t n, uint8_t* d_out_xy112) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_pws || !d_pw_off || !d_out_xy112)) return CAPY_ERR_BAD_ARG;
  return dev_keygen(ctx, dc, st, d_bits, d_pws, d_pw_off, n, d_out_xy112);
}

int capy_ed448_sign_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pws,
                              const uint64_t* d_pw_off, const uint8_t* d_msgs, const uint64_t* d_msg_off, uint64_t n,
                              uint8_t* d_h56, uint8_t* d_z_be56) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_pws || !d_pw_off || !d_msgs || !d_msg_off || !d_h56 || !d_z_be56)) return CAPY_ERR_BAD_ARG;
  return dev_sign(ctx, dc, st, d_bits, d_pws, d_pw_off, d_msgs, d_msg_off, n, d_h56, d_z_be56);
}

int capy_ed448_verify_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pub_xy112,
                                const uint8_t* d_msgs, const uint64_t* d_msg_off, const uint8_t* d_h56,
                                const uint8_t* d_z_be56, uint64_t n, uint8_t* d_ok, int* d_bad_flag) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_pub_xy112 || !d_msgs || !d_msg_off || !d_h56 || !d_z_be56 || !d_ok)) return CAPY_ERR_BAD_ARG;
  return dev_verify(ctx, dc, st, d_bits, d_pub_xy112, d_msgs, d_msg_off, d_h56, d_z_be56, n, d_ok, d_bad_flag);
}

// ---- host-buffer entry points: shard across the ctx devices by item count; inside a device the shard is cut into chunks
// that rotate over the device's streams (run_host_call), so the copies of one chunk run under the kernels of its
// neighbours ----
int capy_ed448_fixed_base_batch(capy_ctx* ctx, const uint8_t* scalars_be56, uint64_t n, uint8_t* out_xy112) {
  if (!ctx || (n && (!scalars_be56 || !out_xy112))) return CAPY_ERR_BAD_ARG;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(nullptr, 1, 0, n, ctx->devs.size(), 0);
  return run_host_call(ctx, shards, ed_chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const uint8_t* d_sc = io.in(scalars_be56, 56);
    uint8_t* d_out = io.out(out_xy112, 112);
    if (io.rc()) return io.rc();
    return dev_fixed_base(ctx, dc, st, d_sc, io.n(), d_out);
  });
}

int capy_ed448_var_base_batch(capy_ctx* ctx, const uint8_t* scalars_be56, const uint8_t* points_xy112, uint64_t n,
                              uint8_t* out_xy112) {
  if (!ctx || (n && (!scalars_be56 || !points_xy112 || !out_xy112))) return CAPY_ERR_BAD_ARG;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(nullptr, 1, 0, n, ctx->devs.size(), 0);
  return run_host_call(ctx, shards, ed_chunks, true, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const uint8_t* d_sc = io.in(scalars_be56, 56);
    const uint8_t* d_pt = io.in(points_xy112, 112);
    uint8_t* d_out = io.out(out_xy112, 112);
    if (io.rc()) return io.rc();
    return dev_var_base(ctx, dc, st, d_sc, d_pt, io.n(), d_out, io.d_flag());
  });
}

int capy_ed448_keygen_batch(capy_ctx* ctx, int d_bits, const uint8_t* pws, const uint64_t* pw_off, uint64_t n,
                            uint8_t* out_xy112) {
  if (!ctx || (n && (!pws || !pw_off || !out_xy112))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(nullptr, 1, 0, n, ctx->devs.size(), 0);
  return run_host_call(ctx, shards, ed_chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(pws, pw_off);
    uint8_t* d_out = io.out(out_xy112, 112);
    if (io.rc()) return io.rc();
    return dev_keygen(ctx, dc, st, d_bits, sp.d_base, sp.d_off, io.n(), d_out);
  });
}

int capy_ed448_sign_batch(capy_ctx* ctx, int d_bits, const uint8_t* pws, const uint64_t* pw_off, const uint8_t* msgs,
                          const uint64_t* msg_off, uint64_t n, uint8_t* h56, uint8_t* z_be56) {
  if (!ctx || (n && (!pws || !pw_off || !msgs || !msg_off || !h56 || !z_be56))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(msg_off, 0, 0, n, ctx->devs.size(), 4096);
  return run_host_call(ctx, shards, ed_chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(pws, pw_off), sm = io.in_packed(msgs, msg_off);
    uint8_t* d_h = io.out(h56, 56);
    uint8_t* d_z = io.out(z_be56, 56);
    if (io.rc()) return io.rc();
    return dev_sign(ctx, dc, st, d_bits, sp.d_base, sp.d_off, sm.d_base, sm.d_off, io.n(), d_h, d_z);
  });
}

int capy_ed448_verify_batch(capy_ctx* ctx, int d_bits, const uint8_t* pub_xy112, const uint8_t* msgs,
                            const uint64_t* msg_off, const uint8_t* h56, const uint8_t* z_be56, uint64_t n, uint8_t* ok) {
  if (!ctx || (n && (!pub_xy112 || !msgs || !msg_off || !h56 || !z_be56 || !ok))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(msg_off, 0, 0, n, ctx->devs.size(), 4096);
  return run_host_call(ctx, shards, ed_chunks, true, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sm = io.in_packed(msgs, msg_off);
    const uint8_t* d_pub = io.in(pub_xy112, 112);
    const uint8_t* d_h = io.in(h56, 56);
    const uint8_t* d_z = io.in(z_be56, 56);
    uint8_t* d_ok = io.out(ok, 1);
    if (io.rc()) return io.rc();
    return dev_verify(ctx, dc, st, d_bits, d_pub, sm.d_base, sm.d_off, d_h, d_z, io.n(), d_ok, io.d_flag());
  });
}

int capy_ed448_verify_prepared_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const capy_ed448_pub* key,
                                         const uint8_t* d_msgs, const uint64_t* d_msg_off, const uint8_t* d_h56,
                                         const uint8_t* d_z_be56, uint64_t n, uint8_t* d_ok) {
  if (pub_check(ctx, key)) return CAPY_ERR_BAD_ARG;
  CAPY_DEV_PROLOGUE
  if (n && (!d_msgs || !d_msg_off || !d_h56 || !d_z_be56 || !d_ok)) return CAPY_ERR_BAD_ARG;
  return dev_verify_prepared(ctx, dc, st, d_bits, key, d_msgs, d_msg_off, d_h56, d_z_be56, n, d_ok);
}

int capy_ed448_verify_prepared_batch(capy_ctx* ctx, int d_bits, const capy_ed448_pub* key, const uint8_t* msgs,
                                     const uint64_t* msg_off, const uint8_t* h56, const uint8_t* z_be56, uint64_t n,
                                     uint8_t* ok) {
  if (!ctx || pub_check(ctx, key) || (n && (!msgs || !msg_off || !h56 || !z_be56 || !ok))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(msg_off, 0, 0, n, ctx->devs.size(), 4096);
  return run_host_call(ctx, shards, ed_chunks, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sm = io.in_packed(msgs, msg_off);
    const uint8_t* d_h = io.in(h56, 56);
    const uint8_t* d_z = io.in(z_be56, 56);
    uint8_t* d_ok = io.out(ok, 1);
    if (io.rc()) return io.rc();
    return dev_verify_prepared(ctx, dc, st, d_bits, key, sm.d_base, sm.d_off, d_h, d_z, io.n(), d_ok);
  });
}

int capy_ed448_pub_prepare(capy_ctx* ctx, const uint8_t* pub_xy112, capy_ed448_pub** out_key) {
  if (!out_key) return CAPY_ERR_BAD_ARG;
  *out_key = nullptr;
  if (!ctx || !pub_xy112) return CAPY_ERR_BAD_ARG;
  {  // on the curve?  (the decoding and the test of var_base_kernel)
    uint32_t w[14];
    Fe x, y;
    PtExt p;
    memcpy(w, pub_xy112, 56);
    fe_from_words(x, w);
    memcpy(w, pub_xy112 + 56, 56);
    fe_from_words(y, w);
    if (!pt_from_affine(p, x, y)) return CAPY_ERR_BAD_POINT;
  }
  capy_ed448_pub* key = new (std::nothrow) capy_ed448_pub();
  if (!key) return CAPY_ERR_OOM;
  key->ctx = ctx;
  memcpy(key->xy, pub_xy112, 112);
  const size_t nd = ctx->devs.size();
  for (const DeviceCtx& dc : ctx->devs) key->dev.push_back(dc.dev);
  key->d_xy.assign(nd, nullptr);
  key->d_table.assign(nd, nullptr);
  const std::vector<uint8_t> scalars = pub_table_scalars();
  bool comb = true;
  for (DeviceCtx& dc : ctx->devs) {
    std::lock_guard<std::mutex> lk(*dc.mu);
    DeviceGuard g(dc.dev);
    const int rc = pub_build_device(ctx, dc, scalars, key, &comb);
    if (rc) {
      capy_ed448_pub_free(key);
      return rc;
    }
  }
  key->comb = comb;  // decided on the first device: the others run the same arithmetic
  *out_key = key;
  return CAPY_OK;
}

int capy_ed448_pub_uses_comb(const capy_ed448_pub* key) { return key && key->comb ? 1 : 0; }

void capy_ed448_pub_free(capy_ed448_pub* key) {
  if (!key) return;
  for (size_t k = 0; k < key->dev.size(); k++) {
    DeviceGuard g(key->dev[k]);
    if (key->d_table[k]) cudaFree(key->d_table[k]);  // cudaFree waits for work that still reads it
    if (key->d_xy[k]) cudaFree(key->d_xy[k]);
  }
  delete key;
}

// The front end of verify up to U'.x (per-item keys: dev_verify; a prepared key: dev_verify_prepared), then KMAC streams
// keyed by U'.x with S = "T" (one chunk per device: the states are stored at [l * items + j]).  h and the off-curve flags
// stay with the streams for capy_hasher_verify_final.
int capy_ed448_verify_stream_new(capy_ctx* ctx, int d_bits, const uint8_t* pub_xy112, const capy_ed448_pub* key,
                                 const uint8_t* h56, const uint8_t* z_be56, uint64_t n, capy_hasher** out) {
  if (!out) return CAPY_ERR_BAD_ARG;
  *out = nullptr;
  if (!ctx || !pub_xy112 == !key || (key && pub_check(ctx, key)) || (n && (!h56 || !z_be56))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (d_bits == 224) return CAPY_ERR_BAD_ARG;  // the "T" stream absorbs at the 172-byte rate (Q7): see the header
  capy_hasher* h = nullptr;
  int rc = hasher_create(ctx, d_bits, kVerifyStream, n, &h, 448);
  if (rc || n == 0) {
    *out = h;
    return rc;
  }
  rc = run_host_call(ctx, hasher_shards(h), one_chunk, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    if (io.n() == 0) return CAPY_OK;  // (a device without items)
    const uint8_t* d_pub = pub_xy112 ? io.in(pub_xy112, 112) : nullptr;
    const uint8_t* d_h = io.in(h56, 56);
    const uint8_t* d_z = io.in(z_be56, 56);
    if (io.rc()) return io.rc();
    const int k = dc.index;
    const uint64_t m = io.n();
    VerifyStart vs;
    int r = d_pub ? dev_verify(ctx, dc, st, d_bits, d_pub, nullptr, nullptr, d_h, d_z, m, nullptr, nullptr, &vs)
                  : dev_verify_prepared(ctx, dc, st, d_bits, key, nullptr, nullptr, d_h, d_z, m, nullptr, &vs);
    if (r) return r;
    CAPY_CUDA(ctx, cudaMemcpyAsync(h->d_h[k], d_h, m * 56, cudaMemcpyDeviceToDevice, st));
    if (vs.bad) CAPY_CUDA(ctx, cudaMemcpyAsync(h->d_bad[k], vs.bad, m, cudaMemcpyDeviceToDevice, st));
    KmacPass a(d_bits, "T", m);
    a.job.keys = vs.ux;
    a.job.key_stride = a.job.key_len = 56;
    return launch_kmac_state(ctx, dc, st, a, false, h->d_state[k]);
  });
  if (rc) {
    capy_hasher_free(h);
    return rc;
  }
  *out = h;
  return CAPY_OK;
}

int capy_ed448_ecdh_batch(capy_ctx* ctx, const uint8_t* k_rand56, const uint8_t* pub_xy112, uint64_t n, uint8_t* wx56,
                          uint8_t* z_xy112) {
  if (!ctx || (n && (!k_rand56 || !pub_xy112 || !wx56))) return CAPY_ERR_BAD_ARG;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(nullptr, 1, 0, n, ctx->devs.size(), 0);
  return run_host_call(ctx, shards, ed_chunks, true, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const uint8_t* d_k = io.in(k_rand56, 56);
    const uint8_t* d_pub = io.in(pub_xy112, 112);
    uint8_t* d_wx = io.out(wx56, 56);
    uint8_t* d_z = z_xy112 ? io.out(z_xy112, 112) : nullptr;
    if (io.rc()) return io.rc();
    return dev_ecdh(ctx, dc, st, d_k, d_pub, io.n(), d_wx, d_z, io.d_flag());
  });
}

}  // extern "C"
