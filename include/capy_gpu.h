/*
 * capy_gpu.h -- C ABI of libcapycrypt_gpu: the B200 (sm_100a) batch engine for capyCRYPT's two
 * data-parallel hot paths (Keccak sponge -> SHA3/cSHAKE/KMACXOF; Ed448-Goldilocks scalar
 * multiplication -> keygen / Schnorr sign+verify / ECDH core).
 *
 * The reference (capyCRYPT 0.7.5, pure Rust) has NO plugin or FFI boundary: its operator
 * surface is a set of traits on `Message` plus `KeyPair::new` and `pub fn kmac_xof`.  Every
 * entry point below is the batched form of one of those operators and cites the reference
 * interface it replaces (paths relative to the reference tree).  A `capycrypt::gpu` Rust
 * module binds these with `extern "C"` (see INTEGRATION.md and rust/gpu.rs).
 *
 * Conventions
 *  - plain pointers and sizes only; every call returns an int status (CAPY_OK == 0, errors < 0);
 *    nothing throws or aborts across the boundary.
 *  - the caller owns every buffer.  Host entry points are blocking; host pointers may be
 *    pageable: large pageable buffers are staged through page-locked buffers of the ctx by a few
 *    copy threads (env CAPY_COPY_THREADS, default up to 8) -- about 20 GB/s; memory from
 *    capy_host_alloc goes straight to the DMA engines -- about 47 GB/s.  `_dev` twins take DEVICE
 *    pointers plus a CUDA stream and are asynchronous on that stream.
 *  - batches: `data` is a packed byte array and `off` has n+1 uint64 offsets into it (item i
 *    = data[off[i] .. off[i+1]) ).  `_fixed` variants take one length and a stride instead.
 *  - d_bits is the reference's SecParam (lib.rs:113-135): 224, 256, 384 or 512; anything else
 *    returns CAPY_ERR_BAD_SECPARAM (= OperationError::UnsupportedSecurityParameter).
 *  - results are bit-exact with the reference INCLUDING its documented deviations from
 *    FIPS 202 / SP 800-185 (SURVEY.md App. A, Q1..Q8).
 *  - field elements: 56 bytes little-endian canonical (FieldElement::to_bytes);
 *    scalars: 56 bytes big-endian (aux_functions.rs:102-110); points: affine x || y, 112 bytes.
 *  - deterministic: no RNG inside; nonces are inputs.
 *  - `_dev` calls only enqueue work (ragged batches also read one small summary back to plan their launch).
 *    They share the ctx's device scratch buffers, so the `_dev` calls of one ctx must be issued on ONE stream at a
 *    time; use one ctx per concurrently used stream.
 *  - a ctx may span several GPUs; host entry points shard the batch across them by contiguous
 *    ranges (no collective: items are independent).  Calls on one ctx are serialised by an
 *    internal mutex; distinct ctxs are independent.
 */
#ifndef CAPY_GPU_H
#define CAPY_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CAPY_OK 0
#define CAPY_ERR_BAD_SECPARAM (-1) /* lib.rs:126-134 UnsupportedSecurityParameter */
#define CAPY_ERR_BAD_ARG (-2)
#define CAPY_ERR_CUDA (-3)
#define CAPY_ERR_BAD_POINT (-4) /* an input point is not on the curve */
#define CAPY_ERR_NO_DEVICE (-5)
#define CAPY_ERR_OOM (-6)

/* flags */
#define CAPY_FLAG_NONE 0u
/* ragged batches are processed longest-message-first (device-side counting sort + one tiny D2H sync);
 * this flag keeps the caller's order and makes the _dev call fully asynchronous */
#define CAPY_FLAG_NO_SORT 1u
/* chain-bound ragged batches run their longest messages with two threads per message (the chain of one message
 * advances faster); this flag keeps one thread per message everywhere (A/B measurements) */
#define CAPY_FLAG_NO_PAIR 2u
/* diagnostics: force the number of warp-tier chains that share a warp scheduler (1..3) in a chain-bound ragged batch
 * instead of letting the planner choose: flags |= c << CAPY_FLAG_WARP_COSCHED_SHIFT */
#define CAPY_FLAG_WARP_COSCHED_SHIFT 8

typedef struct capy_ctx capy_ctx;

/* ---- context ---------------------------------------------------------------------------- */
/* devices == NULL && n_devices <= 0: use the current CUDA device only. */
int capy_gpu_init(const int* devices, int n_devices, capy_ctx** out_ctx);
void capy_gpu_destroy(capy_ctx* ctx);
int capy_gpu_device_count(const capy_ctx* ctx);
/* Overwrites every device scratch buffer of the ctx -- and the page-locked host buffers pageable inputs were staged
 * through -- with zeros.  The pipelines keep intermediate secrets there (derived scalars, KMAC key material, staged
 * passwords) until the next call reuses the buffer; the reference does not zeroize either, so this is an extra for
 * callers who want it.  Blocking. */
int capy_gpu_scrub(capy_ctx* ctx);
const char* capy_strerror(int status);
/* last CUDA error text seen by this ctx (for CAPY_ERR_CUDA) */
const char* capy_last_cuda_error(const capy_ctx* ctx);
int capy_version(void);
/* pinned host memory helpers (optional; faster H2D/D2H for the host entry points) */
void* capy_host_alloc(size_t bytes);
void capy_host_free(void* p);
/* Measurement aid: the ceiling of the host <-> device link for this process.  Per repetition one plain cudaMemcpyAsync
 * of in_bytes host -> device and one of out_bytes device -> host, on two streams so the two directions overlap, no
 * kernel; ms_per_rep is device-timed (events).  Buffers from capy_host_alloc give the pinned-memory figure.  bench.py
 * reports the engine's end-to-end throughput as a fraction of this. */
int capy_copy_probe(capy_ctx* ctx, int dev_index, const void* h_in, size_t in_bytes, void* h_out, size_t out_bytes,
                    int reps, double* ms_per_rep);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches evidence) */
uint64_t capy_launch_count(const capy_ctx* ctx);
/* Plan cache for ragged batches.  A ragged sponge call orders its items longest-first and, for chain-bound batches,
 * splits them into tiers; the shape of that launch depends on the length histogram, which the host reads back (two
 * small D2H copies + stream synchronisations).  With the cache enabled the plan of an offsets array is kept, keyed by
 * (device pointer, n, unit), and every later call that passes the same array -- _dev entry points: the caller's device
 * array; cSHAKE / KMAC / AE alike -- launches without touching the host: the call is asynchronous on the caller's
 * stream.  Contract: an offsets array passed again under the same address has not changed.  A stale plan costs speed,
 * never correctness (the work order stays a permutation of the items and any item may run in any tier).  At most 16
 * plans per device (least recently used evicted); enable = 0 drops them.  Off by default. */
int capy_gpu_set_plan_cache(capy_ctx* ctx, int enable);

/* ---- diagnostics: the host-side launch planner of chain-bound ragged sponge batches (no GPU needed) ------- */
/* items_longer_than[k] = number of items whose message has MORE than k whole rate blocks (k < n_bins), n items,
 * the longest with max_blocks blocks, total_blocks in all.  Returns how many of the longest items run with a whole
 * warp per item and how many of the next with two threads per item (DESIGN.md "chain-bound batches"). */
int capy_plan_tiers(const uint32_t* items_longer_than, uint32_t n_bins, uint64_t n, uint32_t max_blocks,
                    uint64_t total_blocks, int sm_count, uint64_t* warp_items, uint64_t* pair_items);
/* same, with the warp-per-item count split by how many such chains share a warp scheduler: warp_items_by_sharing[c - 1]
 * items run c chains per scheduler, c = 1..3 (a warp-tier chain uses a fraction of its scheduler's issue slots; the
 * longest chains get a scheduler to themselves, the next ones share) */
int capy_plan_tiers3(const uint32_t* items_longer_than, uint32_t n_bins, uint64_t n, uint32_t max_blocks,
                     uint64_t total_blocks, int sm_count, uint64_t* warp_items_by_sharing, uint64_t* pair_items);

/* ---- diagnostics: chain cutting of uniform cSHAKE / KMAC batches (no GPU needed) ------------------------------------
 * A uniform batch whose warps fill the schedulers unevenly (2^16 items on 148 SMs = 3.46 warps per scheduler) is run
 * as two dependent jobs in one launch: the first absorbs `cut_after_blocks` blocks of every item and hands the state
 * over, the second finishes (twice the warps, half as long each).  Returns 1 and the cut when the engine would do that
 * for n items that absorb absorb_blocks blocks (after the cached prefix) and run squeeze_extra permutations between
 * squeeze blocks, 0 when the batch is launched as it is. */
int capy_chain_cut(int sm_count, uint64_t n, uint64_t absorb_blocks, uint64_t squeeze_extra, uint64_t* cut_after_blocks);
/* (environment, read at every launch: CAPY_NO_CHAIN_SPLIT=1 launches such batches uncut -- the A/B switch of the probes
 * and of tests/test_chain_split_gpu.py; results are the same bytes either way) */

/* ---- diagnostics: how a ragged sponge batch is divided over the devices of a ctx (no GPU needed) ------------------- */
/* owner[i] = index of the device that hashes item i when capy_sha3_batch runs on a ctx of `parts` devices: the outliers
 * (messages that cost >= 8 x the average, cost = len / unit_bytes + per_item_cost permutations) are dealt out longest
 * first to the least loaded device (LPT over the chains, SURVEY.md 8e), the rest follows in contiguous index ranges that
 * top every device up to the same load. */
int capy_lpt_shares(const uint64_t* off, uint64_t n, uint32_t parts, uint32_t unit_bytes, uint64_t per_item_cost,
                    uint32_t* owner);

/* ---- SHA3-d : SpongeHashable::compute_sha3_hash (sha3/hashable.rs:19-21 -> shake,
 *      sha3/shake_functions.rs:24-32 -> sponge_absorb/squeeze, sha3/sponge.rs:10-34) ------- */
/* digests: n * (d_bits/8) bytes, item-major.  Hashes the ORIGINAL bytes of every message (the
 * reference additionally leaves Message.msg suffixed+padded, quirk Q5; the Rust shim may
 * replicate that append host-side). */
int capy_sha3_batch(capy_ctx* ctx, int d_bits, const uint8_t* data, const uint64_t* off, uint64_t n,
                    uint8_t* digests, uint32_t flags);
int capy_sha3_batch_fixed(capy_ctx* ctx, int d_bits, const uint8_t* data, uint64_t msg_len, uint64_t stride,
                          uint64_t n, uint8_t* digests, uint32_t flags);
int capy_sha3_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_data,
                        const uint64_t* d_off, uint64_t n, uint8_t* d_digests, uint32_t flags);
int capy_sha3_batch_fixed_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_data,
                              uint64_t msg_len, uint64_t stride, uint64_t n, uint8_t* d_digests, uint32_t flags);

/* ---- cSHAKE : cshake (sha3/shake_functions.rs:49-64), capacity = d bits (quirk Q7) ---------- */
/* out: n * (out_bits/8) bytes.  N = S = "" reproduces the reference's quirk Q4. */
int capy_cshake_batch(capy_ctx* ctx, int d_bits, const uint8_t* data, const uint64_t* off, uint64_t n,
                      const uint8_t* fn_name, uint32_t fn_len, const uint8_t* custom, uint32_t custom_len,
                      uint64_t out_bits, uint8_t* out);
int capy_cshake_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_data,
                          const uint64_t* d_off, uint64_t n, const uint8_t* fn_name, uint32_t fn_len,
                          const uint8_t* custom, uint32_t custom_len, uint64_t out_bits, uint8_t* d_out);

/* ---- KMACXOF : pub fn kmac_xof (sha3/shake_functions.rs:79-89); also
 *      SpongeHashable::compute_tagged_hash (sha3/hashable.rs:33-35) with out_bits = d_bits ---- */
/* keys/key_off: per-item keys (packed + n+1 offsets).  out_off == NULL: every item gets
 * out_bits/8 bytes at stride out_bits/8; otherwise item i writes out[out_off[i]..out_off[i+1])
 * (variable-length squeeze, e.g. the keystream shape of sha3/encryptable.rs:41). */
int capy_kmac_xof_batch(capy_ctx* ctx, int d_bits, const uint8_t* keys, const uint64_t* key_off,
                        const uint8_t* data, const uint64_t* off, uint64_t n, const uint8_t* custom,
                        uint32_t custom_len, uint64_t out_bits, const uint64_t* out_off, uint8_t* out);
int capy_kmac_xof_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_keys,
                            const uint64_t* d_key_off, const uint8_t* d_data, const uint64_t* d_off, uint64_t n,
                            const uint8_t* custom, uint32_t custom_len, uint64_t out_bits,
                            const uint64_t* d_out_off, uint8_t* d_out);
/* fixed-size twin: every key is key_len bytes at key_stride, every message msg_len at msg_stride */
int capy_kmac_xof_batch_fixed_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_keys,
                                  uint64_t key_len, uint64_t key_stride, const uint8_t* d_data, uint64_t msg_len,
                                  uint64_t msg_stride, uint64_t n, const uint8_t* custom, uint32_t custom_len,
                                  uint64_t out_bits, uint8_t* d_out);

/* ---- FIPS 202 SHAKE128/256 -- NO reference counterpart (the reference's `shake` is SHA3-d);
 *      provided because BASELINE.json config 2 names SHAKE256; checked against hashlib. ------ */
int capy_fips_shake_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int shake_bits /*128|256*/,
                              const uint8_t* d_data, const uint64_t* d_off, uint64_t n, uint64_t out_bytes,
                              uint8_t* d_out);

/* ---- Ed448 scalar multiplication : `ExtendedPoint * Scalar` of tiny_ed448_goldilocks 0.1.8,
 *      call sites ecc/keypair.rs:44, ecc/signable.rs:48,77, ecc/encryptable.rs:37-38,78 ------- */
/* out[i] = [k_i]G for the exact integer k_i = BE(scalars[56*i..]) (reduced mod r internally,
 * G has order r).  Fixed-base comb, constant-time table scan. */
int capy_ed448_fixed_base_batch(capy_ctx* ctx, const uint8_t* scalars_be56, uint64_t n, uint8_t* out_xy112);
int capy_ed448_fixed_base_batch_dev(capy_ctx* ctx, int dev_index, void* stream, const uint8_t* d_scalars_be56,
                                    uint64_t n, uint8_t* d_out_xy112);
/* out[i] = [k_i]P_i with k_i the exact (unreduced, up to 448-bit) integer (quirk Q10).
 * Returns CAPY_ERR_BAD_POINT if any P_i is off-curve (that item's output is all zero). */
int capy_ed448_var_base_batch(capy_ctx* ctx, const uint8_t* scalars_be56, const uint8_t* points_xy112, uint64_t n,
                              uint8_t* out_xy112);
int capy_ed448_var_base_batch_dev(capy_ctx* ctx, int dev_index, void* stream, const uint8_t* d_scalars_be56,
                                  const uint8_t* d_points_xy112, uint64_t n, uint8_t* d_out_xy112,
                                  int* d_bad_flag /* device int, set non-zero on a bad point; may be NULL */);

/* ---- KeyPair::new public-key derivation (ecc/keypair.rs:41-51) ------------------------------- */
/* s = 4 * BE(KMACXOF(pw,"",448,"SK",d)) mod r ; V = [s]G ; out = affine V. */
int capy_ed448_keygen_batch(capy_ctx* ctx, int d_bits, const uint8_t* pws, const uint64_t* pw_off, uint64_t n,
                            uint8_t* out_xy112);
int capy_ed448_keygen_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pws,
                                const uint64_t* d_pw_off, uint64_t n, uint8_t* d_out_xy112);

/* ---- Signable::sign / verify (ecc/signable.rs:40-57, 72-86) ------------------------------------ */
/* sign: h56[i] (56 bytes) and z_be56[i] (56 bytes big-endian, canonical in [0, r)). */
int capy_ed448_sign_batch(capy_ctx* ctx, int d_bits, const uint8_t* pws, const uint64_t* pw_off,
                          const uint8_t* msgs, const uint64_t* msg_off, uint64_t n, uint8_t* h56, uint8_t* z_be56);
int capy_ed448_sign_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pws,
                              const uint64_t* d_pw_off, const uint8_t* d_msgs, const uint64_t* d_msg_off,
                              uint64_t n, uint8_t* d_h56, uint8_t* d_z_be56);
/* verify: ok[i] = 1 iff the signature verifies (Ok(())), 0 = SignatureVerificationFailure.
 * Off-curve public keys give ok = 0 and the call returns CAPY_ERR_BAD_POINT. */
int capy_ed448_verify_batch(capy_ctx* ctx, int d_bits, const uint8_t* pub_xy112, const uint8_t* msgs,
                            const uint64_t* msg_off, const uint8_t* h56, const uint8_t* z_be56, uint64_t n,
                            uint8_t* ok);
int capy_ed448_verify_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pub_xy112,
                                const uint8_t* d_msgs, const uint64_t* d_msg_off, const uint8_t* d_h56,
                                const uint8_t* d_z_be56, uint64_t n, uint8_t* d_ok, int* d_bad_flag);

/* ---- ECDH core of KeyEncryptable (ecc/encryptable.rs:36-38 and :76-78) -------------------------- */
/* k_i = 4 * BE(k_rand56[i]) mod r ; wx56[i] = x([k_i]V_i) ; if z_xy112 != NULL also Z_i = [k_i]G.
 * Decrypt side: pass the nonce points Z_i as `pub` and the secret scalars via capy_ed448_var_base_batch. */
int capy_ed448_ecdh_batch(capy_ctx* ctx, const uint8_t* k_rand56, const uint8_t* pub_xy112, uint64_t n,
                          uint8_t* wx56, uint8_t* z_xy112);

/* ---- Sponge AE : SpongeEncryptable::sha3_encrypt / sha3_decrypt (sha3/encryptable.rs:29-45, 58-83) and the
 *      symmetric half of KEMEncryptable::kem_encrypt / kem_decrypt (kem/encryptable.rs:51-57, 91-104, where
 *      `pw` is the ML-KEM shared secret; ML-KEM itself is out of scope) --------------------------------- */
#define CAPY_AE_SHA3 0 /* customisation strings "S", "SKE", "SKA" */
#define CAPY_AE_KEM 1  /* "S", "KEMKE", "KEMKA" */
/* (ke || ka) = KMACXOF(z_i || pw_i, "", 1024, "S"); tag64[i] = KMACXOF(ka, m_i, 512, KA);
 * ct_i = KMACXOF(ke, "", |m_i|, KE) xor m_i, written at the message's own offsets (|ct| == |m|).
 * nonces: n * nonce_len bytes (the reference draws nonce_len = 512 random BYTES, :31); no RNG inside. */
int capy_sponge_encrypt_batch(capy_ctx* ctx, int d_bits, int variant, const uint8_t* pws, const uint64_t* pw_off,
                              const uint8_t* nonces, uint64_t nonce_len, const uint8_t* msgs, const uint64_t* msg_off,
                              uint64_t n, uint8_t* ct, uint8_t* tag64);
/* ok[i] = 1 for Ok(()); 0 = OperationError::SHA3DecryptionFailure, and out_i is then the ciphertext again
 * (the reference XORs the keystream back, :77-82).  `out` must not alias `ct`. */
int capy_sponge_decrypt_batch(capy_ctx* ctx, int d_bits, int variant, const uint8_t* pws, const uint64_t* pw_off,
                              const uint8_t* nonces, uint64_t nonce_len, const uint8_t* ct, const uint64_t* ct_off,
                              const uint8_t* tag64, uint64_t n, uint8_t* out, uint8_t* ok);
/* device twins; pw_bytes = total bytes in d_pws (sizes the z || pw key buffer) */
int capy_sponge_encrypt_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, int variant, const uint8_t* d_pws,
                                  const uint64_t* d_pw_off, uint64_t pw_bytes, const uint8_t* d_nonces, uint64_t nonce_len,
                                  const uint8_t* d_msgs, const uint64_t* d_msg_off, uint64_t n, uint8_t* d_ct,
                                  uint8_t* d_tag64);
int capy_sponge_decrypt_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, int variant, const uint8_t* d_pws,
                                  const uint64_t* d_pw_off, uint64_t pw_bytes, const uint8_t* d_nonces, uint64_t nonce_len,
                                  const uint8_t* d_ct, const uint64_t* d_ct_off, const uint8_t* d_tag64, uint64_t n,
                                  uint8_t* d_out, uint8_t* d_ok);

/* ---- ECDHIES : KeyEncryptable::key_encrypt / key_decrypt (ecc/encryptable.rs:34-50, 72-94) ---------------- */
/* k_i = 4 * BE(k_rand56[i]) mod r; W = [k]V_i; z_xy112[i] = [k]G (Message.asym_nonce, affine);
 * (ke || ka) = KMACXOF(W.x, "", 896, "PK"); tag56[i] = KMACXOF(ka, m_i, 448, "PKA");
 * ct_i = KMACXOF(ke, "", |m_i|, "PKE") xor m_i.  Off-curve V_i -> CAPY_ERR_BAD_POINT (W.x taken as 0). */
int capy_ed448_key_encrypt_batch(capy_ctx* ctx, int d_bits, const uint8_t* pub_xy112, const uint8_t* k_rand56,
                                 const uint8_t* msgs, const uint64_t* msg_off, uint64_t n, uint8_t* ct, uint8_t* tag56,
                                 uint8_t* z_xy112);
/* s = 4 * BE(KMACXOF(pw, "", 448, "SK")) mod r; W = [s]Z_i; ok[i] = 1 for Ok(()), 0 = KeyDecryptionError with
 * out_i = ciphertext (:88-93).  `out` must not alias `ct`. */
int capy_ed448_key_decrypt_batch(capy_ctx* ctx, int d_bits, const uint8_t* pws, const uint64_t* pw_off,
                                 const uint8_t* z_xy112, const uint8_t* ct, const uint64_t* ct_off, const uint8_t* tag56,
                                 uint64_t n, uint8_t* out, uint8_t* ok);
int capy_ed448_key_encrypt_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pub_xy112,
                                     const uint8_t* d_k_rand56, const uint8_t* d_msgs, const uint64_t* d_msg_off, uint64_t n,
                                     uint8_t* d_ct, uint8_t* d_tag56, uint8_t* d_z_xy112, int* d_bad_flag);
int capy_ed448_key_decrypt_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const uint8_t* d_pws,
                                     const uint64_t* d_pw_off, const uint8_t* d_z_xy112, const uint8_t* d_ct,
                                     const uint64_t* d_ct_off, const uint8_t* d_tag56, uint64_t n, uint8_t* d_out,
                                     uint8_t* d_ok, int* d_bad_flag);

/* ---- Prepared public keys: many verifications against one signer, many encryptions to one recipient ------------------
 * Preparing V builds, on every device of the ctx, the comb table of phi(V) (270 KB per device, the layout of G's
 * table).  Verification then computes [z]G + [h]V as one joint comb (two table walks into one accumulator, no
 * doublings) and key_encrypt computes W = [k]V with a second comb instead of the variable-base ladder.  A key is
 * reused across calls: the preparation (a few ms) pays for itself over all the items verified or encrypted with it.
 * Results are byte for byte those of capy_ed448_verify_batch / capy_ed448_key_encrypt_batch with V repeated n times,
 * for every on-curve V. */
typedef struct capy_ed448_pub capy_ed448_pub;
/* Blocking.  CAPY_ERR_BAD_POINT if V is off the curve (*out_key stays NULL).  A V outside the prime-order subgroup (a
 * torsion component) gets no table: the prepared entry points then run the variable-base pipelines, same bytes. */
int capy_ed448_pub_prepare(capy_ctx* ctx, const uint8_t* pub_xy112, capy_ed448_pub** out_key);
/* 1 = V has a comb table, 0 = the prepared entry points fall back to the variable-base pipelines */
int capy_ed448_pub_uses_comb(const capy_ed448_pub* key);
/* Releases the key's device memory.  NULL is a no-op.  Call before capy_gpu_destroy of its ctx. */
void capy_ed448_pub_free(capy_ed448_pub* key);
/* capy_ed448_verify_batch with pub_xy112[i] = V for every i.  A key prepared by another ctx: CAPY_ERR_BAD_ARG. */
int capy_ed448_verify_prepared_batch(capy_ctx* ctx, int d_bits, const capy_ed448_pub* key, const uint8_t* msgs,
                                     const uint64_t* msg_off, const uint8_t* h56, const uint8_t* z_be56, uint64_t n,
                                     uint8_t* ok);
int capy_ed448_verify_prepared_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits, const capy_ed448_pub* key,
                                         const uint8_t* d_msgs, const uint64_t* d_msg_off, const uint8_t* d_h56,
                                         const uint8_t* d_z_be56, uint64_t n, uint8_t* d_ok);
/* capy_ed448_key_encrypt_batch with pub_xy112[i] = V for every i */
int capy_ed448_key_encrypt_prepared_batch(capy_ctx* ctx, int d_bits, const capy_ed448_pub* key, const uint8_t* k_rand56,
                                          const uint8_t* msgs, const uint64_t* msg_off, uint64_t n, uint8_t* ct,
                                          uint8_t* tag56, uint8_t* z_xy112);
int capy_ed448_key_encrypt_prepared_batch_dev(capy_ctx* ctx, int dev_index, void* stream, int d_bits,
                                              const capy_ed448_pub* key, const uint8_t* d_k_rand56, const uint8_t* d_msgs,
                                              const uint64_t* d_msg_off, uint64_t n, uint8_t* d_ct, uint8_t* d_tag56,
                                              uint8_t* d_z_xy112);

/* ---- Resumable SHA3-d and KMACXOF: messages fed in pieces ------------------------------------------------------------
 * A hasher is a batch of n independent streams, one per item, for one operator: SHA3-d (compute_sha3_hash) or KMACXOF
 * (kmac_xof / compute_tagged_hash, one key per item and one customisation string S for the batch).  Each update appends
 * one piece to every stream (item i: data[off[i] .. off[i+1]), empty pieces allowed); the final returns, byte for byte,
 * what capy_sha3_batch / capy_kmac_xof_batch return for the concatenated pieces (Q1, Q2 and Q3 included).  Nothing is
 * packed or kept whole: the device holds per stream its 200-byte state, up to rate - 1 bytes not yet absorbed and the
 * running length.  So a caller whose data arrives in blocks (files, records, logs) needs no concatenated copy, and
 * with the _dev calls can copy piece k + 1 to the device while piece k is absorbed.
 *  - the items are dealt out over the ctx's devices in equal contiguous ranges when the hasher is created
 *    (capy_hasher_device_range); host calls shard by those ranges, a _dev call covers the items [i0, i1) of its device
 *    (d_off: i1 - i0 + 1 offsets into d_data; d_out_off likewise, absolute offsets into d_out).
 *  - the _dev calls of one hasher go, per device, in order on one stream, under the one-stream-at-a-time rule above.
 *  - after final (or final_dev on a device) the hasher is finished: a later update or final (of those items) returns
 *    CAPY_ERR_BAD_ARG.  A hasher of another ctx: CAPY_ERR_BAD_ARG.  n == 0 gives a hasher whose calls do nothing.
 *  - KMACXOF at d_bits = 224 is refused (CAPY_ERR_BAD_ARG): under quirk Q7 its 172-byte rate is counted by 172 but read
 *    by 168, so which bytes are absorbed depends on the final length (the last 4 x blocks bytes of the stream are never
 *    read) and a resumable stream would have to keep about 2.3 % of every message until the final.  SHA3-224 is fine. */
typedef struct capy_hasher capy_hasher;
/* zeroed streams; blocking */
int capy_sha3_hasher_new(capy_ctx* ctx, int d_bits, uint64_t n, capy_hasher** out);
/* absorbs P | bytepad(encode_string(K_i), w) for every item; blocking */
int capy_kmac_xof_hasher_new(capy_ctx* ctx, int d_bits, const uint8_t* keys, const uint64_t* key_off, uint64_t n,
                             const uint8_t* custom, uint32_t custom_len, capy_hasher** out);
int capy_hasher_device_range(const capy_hasher* h, int dev_index, uint64_t* i0, uint64_t* i1);
/* off: n + 1 offsets into data */
int capy_hasher_update(capy_ctx* ctx, capy_hasher* h, const uint8_t* data, const uint64_t* off);
int capy_hasher_update_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, const uint8_t* d_data,
                           const uint64_t* d_off);
/* SHA3-d: out_bits == d_bits and out_off == NULL, n x d_bits/8 digests.  KMACXOF: as capy_kmac_xof_batch (out_bits for
 * every item, or out_off with n + 1 offsets for per-item lengths). */
int capy_hasher_final(capy_ctx* ctx, capy_hasher* h, uint64_t out_bits, const uint64_t* out_off, uint8_t* out);
int capy_hasher_final_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint64_t out_bits,
                          const uint64_t* d_out_off, uint8_t* d_out);
/* zeroes and releases the hasher's device memory (a KMAC state holds key material).  NULL is a no-op.  Call before
 * capy_gpu_destroy of its ctx. */
void capy_hasher_free(capy_hasher* h);

/* ---- Encrypting and verifying in pieces ------------------------------------------------------------------------------
 * Two more kinds of hasher, for the operators that read their message once.  The concatenated pieces give, byte for
 * byte, what the one-shot calls give.  Sign and the decryptions read their message twice: see "Signing and decrypting
 * in two passes" below.
 *  - encryption streams (sha3_encrypt, the KEM symmetric half, key_encrypt): each stream holds the tag sponge, a KMAC
 *    stream keyed by ka, and the keystream sponge KMACXOF(ke, "", ., KE), whose first |m| bytes do not depend on |m|.
 *    ke || ka is derived on the device and never leaves it.  capy_hasher_encrypt_update writes the ciphertext of each
 *    piece at the piece's own offsets; capy_hasher_final with out_bits = 512 (sponge AE) or 448 (key_encrypt) and no
 *    out_off returns the tags.  capy_hasher_update on an encryption stream: CAPY_ERR_BAD_ARG.
 *  - verification streams: U' = [z]G + [h]V is computed at creation, the message goes through capy_hasher_update, and
 *    capy_hasher_verify_final compares h' with h.  capy_hasher_final on a verification stream: CAPY_ERR_BAD_ARG.
 *  - d_bits = 224 is refused (CAPY_ERR_BAD_ARG) for both kinds: the message is absorbed at the 172-byte KMAC rate, as in
 *    capy_kmac_xof_hasher_new.  The one-shot D224 calls are unaffected.
 *  - a prepared key of another ctx, both or neither of pub_xy112 and key: CAPY_ERR_BAD_ARG. */
/* sponge AE seal streams (variant CAPY_AE_SHA3 | CAPY_AE_KEM); nonces: n * nonce_len bytes; blocking */
int capy_sponge_encrypt_stream_new(capy_ctx* ctx, int d_bits, int variant, const uint8_t* pws, const uint64_t* pw_off,
                                   const uint8_t* nonces, uint64_t nonce_len, uint64_t n, capy_hasher** out);
/* key_encrypt seal streams against n keys pub_xy112 or one prepared key; z_xy112 <- Z_i = [k_i]G; blocking.  An off-curve
 * V_i: CAPY_ERR_BAD_POINT and no stream. */
int capy_ed448_key_encrypt_stream_new(capy_ctx* ctx, int d_bits, const uint8_t* pub_xy112, const capy_ed448_pub* key,
                                      const uint8_t* k_rand56, uint64_t n, uint8_t* z_xy112, capy_hasher** out);
/* verification streams against n keys pub_xy112 or one prepared key; blocking.  An off-curve V_i is reported by the final. */
int capy_ed448_verify_stream_new(capy_ctx* ctx, int d_bits, const uint8_t* pub_xy112, const capy_ed448_pub* key,
                                 const uint8_t* h56, const uint8_t* z_be56, uint64_t n, capy_hasher** out);
/* ct[off[i] .. off[i+1]) = keystream ^ data[off[i] .. off[i+1]); ct may alias data */
int capy_hasher_encrypt_update(capy_ctx* ctx, capy_hasher* h, const uint8_t* data, const uint64_t* off, uint8_t* ct);
int capy_hasher_encrypt_update_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, const uint8_t* d_data,
                                   const uint64_t* d_off, uint8_t* d_ct);
/* ok[i] = 1 iff h' == h and V_i is on the curve; CAPY_ERR_BAD_POINT if any V_i was off the curve (_dev: *d_bad_flag |= 1) */
int capy_hasher_verify_final(capy_ctx* ctx, capy_hasher* h, uint8_t* ok);
int capy_hasher_verify_final_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint8_t* d_ok, int* d_bad_flag);

/* ---- Signing and decrypting in two passes -----------------------------------------------------------------------------
 * Sign and the decryptions read their message twice: sign needs k, from a first pass over the message, before its "T"
 * pass; a decryption must not release plaintext before the tag is checked.  The caller feeds every message twice, cut
 * into pieces any way it likes in each pass (empty pieces allowed), with capy_hasher_next_pass between the passes.  The
 * engine checks that both passes carried the same bytes: without that check a sign pass 2 over other bytes would sign
 * them with the k of pass 1, and two signatures sharing k give the private key away; a decryption would release bytes
 * that were never authenticated.
 *  - sign streams: s = 4 BE(KMACXOF(pw, "", 448, "SK")) mod r per item, then the "N" KMAC stream keyed by BE56(s).  Both
 *    passes take capy_hasher_update.  capy_hasher_next_pass (ok = NULL) closes "N" -> N1, k, U = [k]G, and starts "T"
 *    keyed by U.x and a second "N" stream; pass 2 feeds both.  capy_hasher_sign_final: ok[i] = 1 iff the second "N"
 *    output equals N1, and then (h, z) are those of capy_ed448_sign_batch; ok[i] = 0: h and z of item i are zero bytes
 *    and nothing derived from its k leaves the device.
 *  - decryption streams (sha3_decrypt, the KEM symmetric half, key_decrypt): (ke || ka) is derived on the device as the
 *    one-shot calls do, and the expected tags are taken at creation.  Pass 1 takes the ciphertext through
 *    capy_hasher_update and writes nothing.  capy_hasher_next_pass gives the verdict, ok[i] = 1 iff the tag over the
 *    plaintext matched (NULL allowed).  Pass 2 takes capy_hasher_decrypt_update: the plaintext for items whose verdict was
 *    1, the ciphertext for the others.  capy_hasher_decrypt_final: ok[i] = the verdict && the tag over the plaintext of
 *    pass 2 matched too; treat the plaintext of an item with ok[i] = 0 as unauthenticated.
 *  - key_decrypt: an off-curve Z_i fails its item, and capy_hasher_next_pass and capy_hasher_decrypt_final return
 *    CAPY_ERR_BAD_POINT (_dev: *d_bad_flag |= 1), as capy_ed448_key_decrypt_batch does.
 *  - every call out of order is CAPY_ERR_BAD_ARG: a second next_pass, decrypt_update in pass 1, capy_hasher_update on a
 *    decryption stream in pass 2, a final before next_pass, any call after the final, capy_hasher_final /
 *    verify_final / encrypt_update on these kinds, the calls of this block on the other kinds, a hasher of another ctx.
 *    The pass is kept per device, like the finished state.  A next_pass that fails (e.g. CAPY_ERR_OOM) leaves the
 *    streams of its devices unusable: free them.
 *  - d_bits = 224 is refused (CAPY_ERR_BAD_ARG) as for the other streams; a bad variant: CAPY_ERR_BAD_ARG.
 *  - capy_hasher_free zeroes s, k, N1, the key-derived states and the carries (which hold plaintext). */
/* sign streams, one per password; blocking */
int capy_ed448_sign_stream_new(capy_ctx* ctx, int d_bits, const uint8_t* pws, const uint64_t* pw_off, uint64_t n,
                               capy_hasher** out);
/* sponge AE open streams (variant CAPY_AE_SHA3 | CAPY_AE_KEM); nonces: n * nonce_len bytes; tag64: n * 64; blocking */
int capy_sponge_decrypt_stream_new(capy_ctx* ctx, int d_bits, int variant, const uint8_t* pws, const uint64_t* pw_off,
                                   const uint8_t* nonces, uint64_t nonce_len, const uint8_t* tag64, uint64_t n,
                                   capy_hasher** out);
/* key_decrypt streams: z_xy112 the Z of every message, tag56: n * 56; blocking */
int capy_ed448_key_decrypt_stream_new(capy_ctx* ctx, int d_bits, const uint8_t* pws, const uint64_t* pw_off,
                                      const uint8_t* z_xy112, const uint8_t* tag56, uint64_t n, capy_hasher** out);
/* the end of pass 1 (see above) */
int capy_hasher_next_pass(capy_ctx* ctx, capy_hasher* h, uint8_t* ok);
int capy_hasher_next_pass_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint8_t* d_ok, int* d_bad_flag);
/* decryption pass 2: out[off[i] .. off[i+1]) = the plaintext of ct[off[i] .. off[i+1]), or the ciphertext for an item
 * whose verdict was 0; out may alias ct */
int capy_hasher_decrypt_update(capy_ctx* ctx, capy_hasher* h, const uint8_t* ct, const uint64_t* off, uint8_t* out);
int capy_hasher_decrypt_update_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, const uint8_t* d_ct,
                                   const uint64_t* d_off, uint8_t* d_out);
int capy_hasher_decrypt_final(capy_ctx* ctx, capy_hasher* h, uint8_t* ok);
int capy_hasher_decrypt_final_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint8_t* d_ok, int* d_bad_flag);
int capy_hasher_sign_final(capy_ctx* ctx, capy_hasher* h, uint8_t* h56, uint8_t* z_be56, uint8_t* ok);
int capy_hasher_sign_final_dev(capy_ctx* ctx, capy_hasher* h, int dev_index, void* stream, uint8_t* d_h56, uint8_t* d_z_be56,
                               uint8_t* d_ok);

#ifdef __cplusplus
}
#endif
#endif /* CAPY_GPU_H */
