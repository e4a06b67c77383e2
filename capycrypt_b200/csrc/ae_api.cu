// ae_api.cu -- authenticated-encryption compositions over the two hot paths (SURVEY.md 8f, rows N2 and N3).
//
//   sponge AE   SpongeEncryptable::sha3_encrypt / sha3_decrypt     sha3/encryptable.rs:29-45, 58-83
//               symmetric half of KEMEncryptable::kem_encrypt/...  kem/encryptable.rs:51-57, 91-104
//   ECDHIES     KeyEncryptable::key_encrypt / key_decrypt          ecc/encryptable.rs:34-50, 72-94
//
// Both are a key derivation followed by the same two long KMACXOF passes:
//   (ke || ka) <- KMACXOF(secret, "", 2*klen, S0)
//   t          <- KMACXOF(ka, m, tag_bits, S_KA)             over the PLAINTEXT
//   c          <- KMACXOF(ke, "", |m|, S_KE) xor m           keystream, squeezed straight into the XOR
// Decrypt recomputes t' over the recovered plaintext and, on mismatch, hands the ciphertext back unchanged
// (the reference XORs the keystream a second time, encryptable.rs:77-82).  No RNG inside: nonces are inputs.
#include "ed448_kernels.h"
#include "hostbatch.h"

namespace capy {

// keys[i] = nonce_i || pw_i, key_off[i] = i * nonce_len + (pw_off[i] - pw_off[0])   (z.clone(); extend(pw), :33-34)
// one warp per item
__global__ void __launch_bounds__(256) ae_concat_kernel(const uint8_t* __restrict__ nonces, uint64_t nonce_len,
                                                        const uint8_t* __restrict__ pws, const uint64_t* __restrict__ pw_off,
                                                        uint8_t* __restrict__ keys, uint64_t* __restrict__ key_off, uint64_t n) {
  const uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  if (i >= n) return;
  const uint64_t p0 = pw_off[0], a = pw_off[i], b = pw_off[i + 1];
  const uint64_t o = i * nonce_len + (a - p0);
  if (lane == 0) {
    key_off[i] = o;
    if (i + 1 == n) key_off[n] = o + nonce_len + (b - a);
  }
  for (uint64_t k = lane; k < nonce_len; k += 32) keys[o + k] = nonces[i * nonce_len + k];
  for (uint64_t k = lane; k < b - a; k += 32) keys[o + nonce_len + k] = pws[a + k];
}

// ok[i] = (t'_i == t_i) [&& !bad[i]]; on failure the output buffer of item i gets the ciphertext back.
// one warp per item
__global__ void __launch_bounds__(256) ae_finish_kernel(const uint8_t* __restrict__ t_new, const uint8_t* __restrict__ t_in,
                                                        uint32_t tag_bytes, const uint8_t* __restrict__ bad,
                                                        const uint8_t* __restrict__ ct, const uint64_t* __restrict__ off,
                                                        uint8_t* __restrict__ out, uint8_t* __restrict__ ok, uint64_t n) {
  const uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  if (i >= n) return;
  uint32_t diff = 0;
  for (uint32_t k = lane; k < tag_bytes; k += 32) diff |= (uint32_t)(t_new[i * tag_bytes + k] ^ t_in[i * tag_bytes + k]);
  if (bad && bad[i]) diff = 1;
  const bool good = !__any_sync(0xffffffffu, diff != 0);
  if (lane == 0) ok[i] = good ? 1 : 0;
  if (!good && out != ct) {
    const uint64_t a = off[i], b = off[i + 1];
    for (uint64_t k = a + lane; k < b; k += 32) out[k] = ct[k];
  }
}

struct AeCore {
  int d;
  const uint8_t* keymat;  // n x (2 * klen): ke || ka
  uint32_t klen;
  const char* ke_custom;
  const char* ka_custom;
  uint32_t tag_bytes;
};

// t = KMACXOF(ka, m, tag, KA) ; c = KMACXOF(ke, "", |m|, KE) ^ m.  `ct` may alias `msgs` (in place): then the tag
// pass has to finish before the keystream overwrites the message; otherwise the two passes are independent and go
// out as ONE launch (launch_kmac_xof2: twice the warps, so the last wave of the grid is full).
static int dev_ae_seal(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const AeCore& c, const uint8_t* msgs,
                       const uint64_t* off, uint64_t n, uint8_t* ct, uint8_t* tag) {
  KmacPass a(c.d, c.ka_custom, n);
  a.job.keys = c.keymat + c.klen;
  a.job.key_len = c.klen;
  a.job.key_stride = 2ull * c.klen;
  a.job.data = msgs;
  a.job.off = off;
  a.job.out_bytes = a.job.out_stride = c.tag_bytes;
  a.job.out = tag;
  KmacPass k(c.d, c.ke_custom, n);
  k.job.keys = c.keymat;
  k.job.key_len = c.klen;
  k.job.key_stride = 2ull * c.klen;
  k.job.out_off = off;
  k.job.out = ct;
  k.job.xor_in = msgs;
  if (ct != msgs) return launch_kmac_xof2(ctx, dc, st, a, k);
  int rc = launch_kmac_xof(ctx, dc, st, a);
  if (rc) return rc;
  return launch_kmac_xof(ctx, dc, st, k);
}

// m = KMACXOF(ke, "", |c|, KE) ^ c ; t' = KMACXOF(ka, m, tag, KA) ; compare ; restore on failure.
static int dev_ae_open(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const AeCore& c, const uint8_t* ct,
                       const uint64_t* off, const uint8_t* tag, const uint8_t* bad, uint64_t n, uint8_t* out, uint8_t* ok,
                       uint8_t* t_new) {
  if (out == ct) return CAPY_ERR_BAD_ARG;  // the ciphertext must survive for the restore-on-failure path
  KmacPass k(c.d, c.ke_custom, n);
  k.job.keys = c.keymat;
  k.job.key_len = c.klen;
  k.job.key_stride = 2ull * c.klen;
  k.job.out_off = off;
  k.job.out = out;
  k.job.xor_in = ct;
  KmacPass a(c.d, c.ka_custom, n);
  a.job.keys = c.keymat + c.klen;
  a.job.key_len = c.klen;
  a.job.key_stride = 2ull * c.klen;
  a.job.data = out;
  a.job.off = off;
  a.job.out_bytes = a.job.out_stride = c.tag_bytes;
  a.job.out = t_new;
  // the tag pass reads what the keystream pass writes: dependent jobs of one launch when the batch is large enough
  int rc = launch_kmac_xof_dep(ctx, dc, st, k, a);
  if (rc) return rc;
  ae_finish_kernel<<<grid_for(n * 32, 256), 256, 0, st>>>(t_new, tag, c.tag_bytes, bad, ct, off, out, ok, n);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  return CAPY_OK;
}

static bool ae_customs(int variant, const char** ke, const char** ka) {
  if (variant == CAPY_AE_SHA3) {
    *ke = "SKE";  // sha3/encryptable.rs:41
    *ka = "SKA";  // :39
    return true;
  }
  if (variant == CAPY_AE_KEM) {
    *ke = "KEMKE";  // kem/encryptable.rs:56
    *ka = "KEMKA";  // :54
    return true;
  }
  return false;
}

// (ke || ka) <- KMACXOF(z || pw, "", 1024, "S")   sha3/encryptable.rs:33-37
static int dev_sponge_keymat(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* pws, const uint64_t* pw_off,
                             uint64_t pw_bytes, const uint8_t* nonces, uint64_t nonce_len, uint64_t n, uint8_t** keymat_out) {
  CAPY_SCRATCH(keys, uint8_t, kAeKeys, n * nonce_len + pw_bytes + 16);
  CAPY_SCRATCH(koff, uint64_t, kAeKeyOff, (n + 1) * 8);
  CAPY_SCRATCH(keymat, uint8_t, kAeKeyMat, n * 128);
  ae_concat_kernel<<<grid_for(n * 32, 256), 256, 0, st>>>(nonces, nonce_len, pws, pw_off, keys, koff, n);
  ctx->launches++;
  CAPY_CUDA(ctx, cudaGetLastError());
  KmacPass a(d, "S", n);
  a.job.keys = keys;
  a.job.key_off = koff;
  a.job.out_bytes = a.job.out_stride = 128;
  a.job.out = keymat;
  a.no_sort = true;
  *keymat_out = keymat;
  return launch_kmac_xof(ctx, dc, st, a);
}

static int dev_sponge_encrypt(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, int variant, const uint8_t* pws,
                              const uint64_t* pw_off, uint64_t pw_bytes, const uint8_t* nonces, uint64_t nonce_len,
                              const uint8_t* msgs, const uint64_t* off, uint64_t n, uint8_t* ct, uint8_t* tag) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  AeCore c{};
  if (!ae_customs(variant, &c.ke_custom, &c.ka_custom)) return CAPY_ERR_BAD_ARG;
  if (n == 0) return CAPY_OK;
  uint8_t* keymat;
  int rc = dev_sponge_keymat(ctx, dc, st, d, pws, pw_off, pw_bytes, nonces, nonce_len, n, &keymat);
  if (rc) return rc;
  c.d = d;
  c.keymat = keymat;
  c.klen = 64;       // ke_ka.split_at(64)
  c.tag_bytes = 64;  // 512 bits
  return dev_ae_seal(ctx, dc, st, c, msgs, off, n, ct, tag);
}

static int dev_sponge_decrypt(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, int variant, const uint8_t* pws,
                              const uint64_t* pw_off, uint64_t pw_bytes, const uint8_t* nonces, uint64_t nonce_len,
                              const uint8_t* ct, const uint64_t* off, const uint8_t* tag, uint64_t n, uint8_t* out,
                              uint8_t* ok) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  AeCore c{};
  if (!ae_customs(variant, &c.ke_custom, &c.ka_custom)) return CAPY_ERR_BAD_ARG;
  if (n == 0) return CAPY_OK;
  uint8_t* keymat;
  int rc = dev_sponge_keymat(ctx, dc, st, d, pws, pw_off, pw_bytes, nonces, nonce_len, n, &keymat);
  if (rc) return rc;
  CAPY_SCRATCH(t_new, uint8_t, kAeTNew, n * 64);
  c.d = d;
  c.keymat = keymat;
  c.klen = 64;
  c.tag_bytes = 64;
  return dev_ae_open(ctx, dc, st, c, ct, off, tag, nullptr, n, out, ok, t_new);
}

// (ke || ka) <- KMACXOF(W.x, "", 896, "PK")   ecc/encryptable.rs:40-41, 80-81
static int dev_ecdhies_keymat(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* wx, uint64_t n,
                              uint8_t** keymat_out) {
  CAPY_SCRATCH(keymat, uint8_t, kAeKeyMat, n * 112);
  KmacPass a(d, "PK", n);
  a.job.keys = wx;
  a.job.key_stride = a.job.key_len = 56;
  a.job.out_bytes = a.job.out_stride = 112;
  a.job.out = keymat;
  *keymat_out = keymat;
  return launch_kmac_xof(ctx, dc, st, a);
}

static AeCore ecdhies_core(int d, const uint8_t* keymat) {
  AeCore c{};
  c.d = d;
  c.keymat = keymat;
  c.klen = 56;  // split_at(len / 2)
  c.ke_custom = "PKE";
  c.ka_custom = "PKA";
  c.tag_bytes = 56;  // 448 bits
  return c;
}

// Z = [k]G (:38) with kw = k in SoA words ; (ke || ka) from W.x ; tag and ciphertext (:40-48).  With keymat_out, no
// message: (ke || ka) is handed back for an encryption stream instead.
static int key_encrypt_finish(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint32_t* kw, const uint8_t* wx,
                              const uint8_t* msgs, const uint64_t* off, uint64_t n, uint8_t* ct, uint8_t* tag, uint8_t* z_xy,
                              uint8_t** keymat_out) {
  CAPY_SCRATCH(proj, uint32_t, kAeProj, n * 256);
  int rc = launch_fixed_base(ctx, dc, st, kw, proj, n, true);
  if (rc) return rc;
  rc = launch_to_affine(ctx, st, proj, n, 0, nullptr, z_xy);
  if (rc) return rc;
  uint8_t* keymat;
  rc = dev_ecdhies_keymat(ctx, dc, st, d, wx, n, &keymat);
  if (rc) return rc;
  if (keymat_out) {
    *keymat_out = keymat;
    return CAPY_OK;
  }
  return dev_ae_seal(ctx, dc, st, ecdhies_core(d, keymat), msgs, off, n, ct, tag);
}

static int dev_key_encrypt(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* pub, const uint8_t* k_rand,
                           const uint8_t* msgs, const uint64_t* off, uint64_t n, uint8_t* ct, uint8_t* tag, uint8_t* z_xy,
                           int* d_bad_flag, uint8_t** keymat_out = nullptr) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(proj, uint32_t, kAeProj, n * 256);
  CAPY_SCRATCH(bad, uint8_t, kAeBad, n);
  CAPY_SCRATCH(wx, uint8_t, kAeWx, n * 56);
  CAPY_SCRATCH(kw, uint32_t, kAeKw, n * 56);
  // k = 4 * BE(rand) mod r ; W = [k]V (:36-37)
  int rc = launch_var_base(ctx, dc, st, k_rand, 1, pub, nullptr, proj, bad, n, true);
  if (rc) return rc;
  rc = launch_to_affine(ctx, st, proj, n, 1, bad, wx);
  if (rc) return rc;
  rc = launch_scalar_prep(ctx, st, k_rand, 1, kw, nullptr, n);
  if (rc) return rc;
  rc = key_encrypt_finish(ctx, dc, st, d, kw, wx, msgs, off, n, ct, tag, z_xy, keymat_out);
  if (rc) return rc;
  return d_bad_flag ? launch_any_bad(ctx, st, bad, d_bad_flag, n) : CAPY_OK;
}

// W = [k]V for a prepared V through V's comb table (k is secret: constant-time scan), then as dev_key_encrypt
static int dev_key_encrypt_prepared(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const capy_ed448_pub* key,
                                    const uint8_t* k_rand, const uint8_t* msgs, const uint64_t* off, uint64_t n, uint8_t* ct,
                                    uint8_t* tag, uint8_t* z_xy, uint8_t** keymat_out = nullptr) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  const uint32_t* v_table = key->d_table[dc.index];
  if (!v_table) {  // V has a torsion component: the variable-base pipeline with V repeated
    CAPY_SCRATCH(pub, uint8_t, kEdPubRep, n * 112);
    const int rc = broadcast_point(ctx, st, key->d_xy[dc.index], pub, n);
    if (rc) return rc;
    return dev_key_encrypt(ctx, dc, st, d, pub, k_rand, msgs, off, n, ct, tag, z_xy, nullptr, keymat_out);
  }
  CAPY_SCRATCH(proj, uint32_t, kAeProj, n * 256);
  CAPY_SCRATCH(wx, uint8_t, kAeWx, n * 56);
  CAPY_SCRATCH(kw, uint32_t, kAeKw, n * 56);
  // k = 4 * BE(rand) mod r ; W = [k]V (:36-37)
  int rc = launch_scalar_prep(ctx, st, k_rand, 1, kw, nullptr, n);
  if (rc) return rc;
  rc = launch_fixed_base(ctx, dc, st, kw, proj, n, true, v_table);
  if (rc) return rc;
  rc = launch_to_affine(ctx, st, proj, n, 1, nullptr, wx);
  if (rc) return rc;
  return key_encrypt_finish(ctx, dc, st, d, kw, wx, msgs, off, n, ct, tag, z_xy, keymat_out);
}

static int dev_key_decrypt(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, int d, const uint8_t* pws, const uint64_t* pw_off,
                           const uint8_t* z_xy, const uint8_t* ct, const uint64_t* off, const uint8_t* tag, uint64_t n,
                           uint8_t* out, uint8_t* ok, int* d_bad_flag) {
  if (!valid_secparam(d)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  CAPY_SCRATCH(proj, uint32_t, kAeProj, n * 256);
  CAPY_SCRATCH(bad, uint8_t, kAeBad, n);
  CAPY_SCRATCH(wx, uint8_t, kAeWx, n * 56);
  CAPY_SCRATCH(sk, uint8_t, kAeSk, n * 56);
  CAPY_SCRATCH(t_new, uint8_t, kAeTNew, n * 56);
  // s = 4 * BE(KMACXOF(pw, "", 448, "SK")) mod r (:74-75)
  KmacPass a(d, "SK", n);
  a.job.keys = pws;
  a.job.key_off = pw_off;
  a.job.out_bytes = a.job.out_stride = 56;
  a.job.out = sk;
  a.no_sort = true;
  int rc = launch_kmac_xof(ctx, dc, st, a);
  if (rc) return rc;
  // W = [s]Z (:76)
  rc = launch_var_base(ctx, dc, st, sk, 1, z_xy, nullptr, proj, bad, n, true);
  if (rc) return rc;
  rc = launch_to_affine(ctx, st, proj, n, 1, bad, wx);
  if (rc) return rc;
  uint8_t* keymat;
  rc = dev_ecdhies_keymat(ctx, dc, st, d, wx, n, &keymat);
  if (rc) return rc;
  rc = dev_ae_open(ctx, dc, st, ecdhies_core(d, keymat), ct, off, tag, bad, n, out, ok, t_new);
  if (rc) return rc;
  return d_bad_flag ? launch_any_bad(ctx, st, bad, d_bad_flag, n) : CAPY_OK;
}

// The two sponges of an encryption stream (capy_hasher) from (ke || ka) on the device, for the items of device dc: the tag
// stream KMAC(ka, ., KA) after P | KB, and the keystream KMAC(ke, "", ., KE) at the start of its first squeeze block
static int ae_stream_start(capy_ctx* ctx, DeviceCtx& dc, cudaStream_t st, const AeCore& c, capy_hasher* h, uint64_t n) {
  KmacPass a(c.d, c.ka_custom, n);
  a.job.keys = c.keymat + c.klen;
  a.job.key_len = c.klen;
  a.job.key_stride = 2ull * c.klen;
  int rc = launch_kmac_state(ctx, dc, st, a, false, h->d_state[dc.index]);
  if (rc) return rc;
  KmacPass k(c.d, c.ke_custom, n);
  k.job.keys = c.keymat;
  k.job.key_len = c.klen;
  k.job.key_stride = 2ull * c.klen;
  return launch_kmac_state(ctx, dc, st, k, true, h->d_ks_state[dc.index]);
}

}  // namespace capy

using namespace capy;

extern "C" {

// =================================================================================================
// sponge AE
// =================================================================================================
int capy_sponge_encrypt_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, int variant, const uint8_t* d_pws,
                                  const uint64_t* d_pw_off, uint64_t pw_bytes, const uint8_t* d_nonces, uint64_t nonce_len,
                                  const uint8_t* d_msgs, const uint64_t* d_msg_off, uint64_t n, uint8_t* d_ct,
                                  uint8_t* d_tag64) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_pws || !d_pw_off || !d_nonces || !d_msgs || !d_msg_off || !d_ct || !d_tag64)) return CAPY_ERR_BAD_ARG;
  return dev_sponge_encrypt(ctx, dc, st, d_bits, variant, d_pws, d_pw_off, pw_bytes, d_nonces, nonce_len, d_msgs, d_msg_off, n,
                            d_ct, d_tag64);
}

int capy_sponge_decrypt_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, int variant, const uint8_t* d_pws,
                                  const uint64_t* d_pw_off, uint64_t pw_bytes, const uint8_t* d_nonces, uint64_t nonce_len,
                                  const uint8_t* d_ct, const uint64_t* d_ct_off, const uint8_t* d_tag64, uint64_t n,
                                  uint8_t* d_out, uint8_t* d_ok) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_pws || !d_pw_off || !d_nonces || !d_ct || !d_ct_off || !d_tag64 || !d_out || !d_ok)) return CAPY_ERR_BAD_ARG;
  return dev_sponge_decrypt(ctx, dc, st, d_bits, variant, d_pws, d_pw_off, pw_bytes, d_nonces, nonce_len, d_ct, d_ct_off,
                            d_tag64, n, d_out, d_ok);
}

int capy_sponge_encrypt_batch(capy_ctx* ctx, int d_bits, int variant, const uint8_t* pws, const uint64_t* pw_off,
                              const uint8_t* nonces, uint64_t nonce_len, const uint8_t* msgs, const uint64_t* msg_off,
                              uint64_t n, uint8_t* ct, uint8_t* tag64) {
  if (!ctx || (n && (!pws || !pw_off || !nonces || !msgs || !msg_off || !ct || !tag64))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (variant != CAPY_AE_SHA3 && variant != CAPY_AE_KEM) return CAPY_ERR_BAD_ARG;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(msg_off, 0, 0, n, ctx->devs.size(), 2048);
  return run_host_call(ctx, shards, one_chunk, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(pws, pw_off), sm = io.in_packed(msgs, msg_off);
    const uint8_t* d_nonce = io.in(nonces, nonce_len);
    uint8_t* d_ct = io.out_packed(ct, msg_off);
    uint8_t* d_tag = io.out(tag64, 64);
    if (io.rc()) return io.rc();
    return dev_sponge_encrypt(ctx, dc, st, d_bits, variant, sp.d_base, sp.d_off, pw_off[io.i1()] - pw_off[io.i0()], d_nonce,
                              nonce_len, sm.d_base, sm.d_off, io.n(), d_ct, d_tag);
  });
}

int capy_sponge_decrypt_batch(capy_ctx* ctx, int d_bits, int variant, const uint8_t* pws, const uint64_t* pw_off,
                              const uint8_t* nonces, uint64_t nonce_len, const uint8_t* ct, const uint64_t* ct_off,
                              const uint8_t* tag64, uint64_t n, uint8_t* out, uint8_t* ok) {
  if (!ctx || (n && (!pws || !pw_off || !nonces || !ct || !ct_off || !tag64 || !out || !ok))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (variant != CAPY_AE_SHA3 && variant != CAPY_AE_KEM) return CAPY_ERR_BAD_ARG;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(ct_off, 0, 0, n, ctx->devs.size(), 2048);
  return run_host_call(ctx, shards, one_chunk, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(pws, pw_off), sc = io.in_packed(ct, ct_off);
    const uint8_t* d_nonce = io.in(nonces, nonce_len);
    const uint8_t* d_tag = io.in(tag64, 64);
    uint8_t* d_out = io.out_packed(out, ct_off);
    uint8_t* d_ok = io.out(ok, 1);
    if (io.rc()) return io.rc();
    return dev_sponge_decrypt(ctx, dc, st, d_bits, variant, sp.d_base, sp.d_off, pw_off[io.i1()] - pw_off[io.i0()], d_nonce,
                              nonce_len, sc.d_base, sc.d_off, d_tag, io.n(), d_out, d_ok);
  });
}

// =================================================================================================
// ECDHIES
// =================================================================================================
int capy_ed448_key_encrypt_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pub_xy112,
                                     const uint8_t* d_k_rand56, const uint8_t* d_msgs, const uint64_t* d_msg_off, uint64_t n,
                                     uint8_t* d_ct, uint8_t* d_tag56, uint8_t* d_z_xy112, int* d_bad_flag) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_pub_xy112 || !d_k_rand56 || !d_msgs || !d_msg_off || !d_ct || !d_tag56 || !d_z_xy112)) return CAPY_ERR_BAD_ARG;
  return dev_key_encrypt(ctx, dc, st, d_bits, d_pub_xy112, d_k_rand56, d_msgs, d_msg_off, n, d_ct, d_tag56, d_z_xy112,
                         d_bad_flag);
}

int capy_ed448_key_decrypt_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pws,
                                     const uint64_t* d_pw_off, const uint8_t* d_z_xy112, const uint8_t* d_ct,
                                     const uint64_t* d_ct_off, const uint8_t* d_tag56, uint64_t n, uint8_t* d_out,
                                     uint8_t* d_ok, int* d_bad_flag) {
  CAPY_DEV_PROLOGUE
  if (n && (!d_pws || !d_pw_off || !d_z_xy112 || !d_ct || !d_ct_off || !d_tag56 || !d_out || !d_ok)) return CAPY_ERR_BAD_ARG;
  return dev_key_decrypt(ctx, dc, st, d_bits, d_pws, d_pw_off, d_z_xy112, d_ct, d_ct_off, d_tag56, n, d_out, d_ok, d_bad_flag);
}

int capy_ed448_key_encrypt_batch(capy_ctx* ctx, int d_bits, const uint8_t* pub_xy112, const uint8_t* k_rand56,
                                 const uint8_t* msgs, const uint64_t* msg_off, uint64_t n, uint8_t* ct, uint8_t* tag56,
                                 uint8_t* z_xy112) {
  if (!ctx || (n && (!pub_xy112 || !k_rand56 || !msgs || !msg_off || !ct || !tag56 || !z_xy112))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(msg_off, 0, 0, n, ctx->devs.size(), 16384);
  return run_host_call(ctx, shards, one_chunk, true, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sm = io.in_packed(msgs, msg_off);
    const uint8_t* d_pub = io.in(pub_xy112, 112);
    const uint8_t* d_k = io.in(k_rand56, 56);
    uint8_t* d_ct = io.out_packed(ct, msg_off);
    uint8_t* d_tag = io.out(tag56, 56);
    uint8_t* d_z = io.out(z_xy112, 112);
    if (io.rc()) return io.rc();
    return dev_key_encrypt(ctx, dc, st, d_bits, d_pub, d_k, sm.d_base, sm.d_off, io.n(), d_ct, d_tag, d_z, io.d_flag());
  });
}

int capy_ed448_key_encrypt_prepared_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits,
                                              const capy_ed448_pub* key, const uint8_t* d_k_rand56, const uint8_t* d_msgs,
                                              const uint64_t* d_msg_off, uint64_t n, uint8_t* d_ct, uint8_t* d_tag56,
                                              uint8_t* d_z_xy112) {
  if (pub_check(ctx, key)) return CAPY_ERR_BAD_ARG;
  CAPY_DEV_PROLOGUE
  if (n && (!d_k_rand56 || !d_msgs || !d_msg_off || !d_ct || !d_tag56 || !d_z_xy112)) return CAPY_ERR_BAD_ARG;
  return dev_key_encrypt_prepared(ctx, dc, st, d_bits, key, d_k_rand56, d_msgs, d_msg_off, n, d_ct, d_tag56, d_z_xy112);
}

int capy_ed448_key_encrypt_prepared_batch(capy_ctx* ctx, int d_bits, const capy_ed448_pub* key, const uint8_t* k_rand56,
                                          const uint8_t* msgs, const uint64_t* msg_off, uint64_t n, uint8_t* ct,
                                          uint8_t* tag56, uint8_t* z_xy112) {
  if (!ctx || pub_check(ctx, key) || (n && (!k_rand56 || !msgs || !msg_off || !ct || !tag56 || !z_xy112)))
    return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(msg_off, 0, 0, n, ctx->devs.size(), 16384);
  return run_host_call(ctx, shards, one_chunk, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sm = io.in_packed(msgs, msg_off);
    const uint8_t* d_k = io.in(k_rand56, 56);
    uint8_t* d_ct = io.out_packed(ct, msg_off);
    uint8_t* d_tag = io.out(tag56, 56);
    uint8_t* d_z = io.out(z_xy112, 112);
    if (io.rc()) return io.rc();
    return dev_key_encrypt_prepared(ctx, dc, st, d_bits, key, d_k, sm.d_base, sm.d_off, io.n(), d_ct, d_tag, d_z);
  });
}

int capy_ed448_key_decrypt_batch(capy_ctx* ctx, int d_bits, const uint8_t* pws, const uint64_t* pw_off,
                                 const uint8_t* z_xy112, const uint8_t* ct, const uint64_t* ct_off, const uint8_t* tag56,
                                 uint64_t n, uint8_t* out, uint8_t* ok) {
  if (!ctx || (n && (!pws || !pw_off || !z_xy112 || !ct || !ct_off || !tag56 || !out || !ok))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (n == 0) return CAPY_OK;
  auto shards = split_items(ct_off, 0, 0, n, ctx->devs.size(), 16384);
  return run_host_call(ctx, shards, one_chunk, true, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    const StagedPacked sp = io.in_packed(pws, pw_off), sc = io.in_packed(ct, ct_off);
    const uint8_t* d_z = io.in(z_xy112, 112);
    const uint8_t* d_tag = io.in(tag56, 56);
    uint8_t* d_out = io.out_packed(out, ct_off);
    uint8_t* d_ok = io.out(ok, 1);
    if (io.rc()) return io.rc();
    return dev_key_decrypt(ctx, dc, st, d_bits, sp.d_base, sp.d_off, d_z, sc.d_base, sc.d_off, d_tag, io.n(), d_out, d_ok,
                           io.d_flag());
  });
}

// =================================================================================================
// encryption streams: the plaintext fed in pieces (capy_hasher_encrypt_update), the tag from capy_hasher_final
// =================================================================================================
// one chunk per device: the states are stored at [l * items + j]
int capy_sponge_encrypt_stream_new(capy_ctx* ctx, int d_bits, int variant, const uint8_t* pws, const uint64_t* pw_off,
                                   const uint8_t* nonces, uint64_t nonce_len, uint64_t n, capy_hasher** out) {
  if (!out) return CAPY_ERR_BAD_ARG;
  *out = nullptr;
  AeCore c{};
  if (!ctx || (n && (!pws || !pw_off || !nonces)) || !ae_customs(variant, &c.ke_custom, &c.ka_custom)) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (d_bits == 224) return CAPY_ERR_BAD_ARG;  // the tag stream absorbs at the 172-byte rate (Q7): see the header
  capy_hasher* h = nullptr;
  int rc = hasher_create(ctx, d_bits, kEncryptStream, n, &h, 512);
  if (rc || n == 0) {
    *out = h;
    return rc;
  }
  rc = run_host_call(ctx, hasher_shards(h), one_chunk, false, [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    if (io.n() == 0) return CAPY_OK;  // (a device without items)
    const StagedPacked sp = io.in_packed(pws, pw_off);
    const uint8_t* d_nonce = io.in(nonces, nonce_len);
    if (io.rc()) return io.rc();
    uint8_t* keymat;
    const int r = dev_sponge_keymat(ctx, dc, st, d_bits, sp.d_base, sp.d_off, pw_off[io.i1()] - pw_off[io.i0()], d_nonce,
                                    nonce_len, io.n(), &keymat);
    if (r) return r;
    AeCore cc = c;
    cc.d = d_bits;
    cc.keymat = keymat;
    cc.klen = 64;  // ke_ka.split_at(64)
    return ae_stream_start(ctx, dc, st, cc, h, io.n());
  });
  if (rc) {
    capy_hasher_free(h);
    return rc;
  }
  *out = h;
  return CAPY_OK;
}

int capy_ed448_key_encrypt_stream_new(capy_ctx* ctx, int d_bits, const uint8_t* pub_xy112, const capy_ed448_pub* key,
                                      const uint8_t* k_rand56, uint64_t n, uint8_t* z_xy112, capy_hasher** out) {
  if (!out) return CAPY_ERR_BAD_ARG;
  *out = nullptr;
  if (!ctx || !pub_xy112 == !key || (key && pub_check(ctx, key)) || (n && (!k_rand56 || !z_xy112))) return CAPY_ERR_BAD_ARG;
  if (!valid_secparam(d_bits)) return CAPY_ERR_BAD_SECPARAM;
  if (d_bits == 224) return CAPY_ERR_BAD_ARG;
  capy_hasher* h = nullptr;
  int rc = hasher_create(ctx, d_bits, kEncryptStream, n, &h, 448);
  if (rc || n == 0) {
    *out = h;
    return rc;
  }
  rc = run_host_call(ctx, hasher_shards(h), one_chunk, pub_xy112 != nullptr,
                     [&](DeviceCtx& dc, cudaStream_t st, HostChunk& io) -> int {
    if (io.n() == 0) return CAPY_OK;
    const uint8_t* d_pub = pub_xy112 ? io.in(pub_xy112, 112) : nullptr;
    const uint8_t* d_k = io.in(k_rand56, 56);
    uint8_t* d_z = io.out(z_xy112, 112);
    if (io.rc()) return io.rc();
    uint8_t* keymat;
    const int r = d_pub ? dev_key_encrypt(ctx, dc, st, d_bits, d_pub, d_k, nullptr, nullptr, io.n(), nullptr, nullptr, d_z,
                                          io.d_flag(), &keymat)
                        : dev_key_encrypt_prepared(ctx, dc, st, d_bits, key, d_k, nullptr, nullptr, io.n(), nullptr, nullptr,
                                                   d_z, &keymat);
    if (r) return r;
    return ae_stream_start(ctx, dc, st, ecdhies_core(d_bits, keymat), h, io.n());
  });
  if (rc) {  // CAPY_ERR_BAD_POINT included: no stream for a batch with an off-curve key
    capy_hasher_free(h);
    return rc;
  }
  *out = h;
  return CAPY_OK;
}

}  // extern "C"
