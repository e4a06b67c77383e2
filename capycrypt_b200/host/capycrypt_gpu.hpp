// capycrypt_gpu.hpp -- C++ host-side mirror of capyCRYPT's operator surface for batches, over the C ABI of
// libcapycrypt_gpu (include/capy_gpu.h).  The reference is compiled (Rust) code and the Rust toolchain is
// absent from this image, so the host side above the C ABI is C++ with the reference's names:
//   capycrypt::SecParam        src/lib.rs:113-135        capycrypt::OperationError  src/lib.rs:9-30
//   capycrypt::Message         src/lib.rs:65-94          capycrypt::Signature       src/ecc/signable.rs:17-24
//   capycrypt::KeyPair         src/ecc/keypair.rs:13-51
//   capycrypt::gpu::Engine     batch forms of SpongeHashable (sha3/hashable.rs:7-36), kmac_xof
//                              (sha3/shake_functions.rs:79-89), KeyPair::new, Signable (ecc/signable.rs:12-15),
//                              SpongeEncryptable (sha3/encryptable.rs:7-10), KeyEncryptable (ecc/encryptable.rs:10-13)
// Header-only; link with -lcapycrypt_gpu.  Nothing is computed on the CPU.
#pragma once
#include <array>
#include <random>
#include <cstdint>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/capy_gpu.h"

namespace capycrypt {

enum class OperationError {  // src/lib.rs:9-30 (the variants the hot path can produce)
  UnsupportedSecurityParameter,
  SignatureVerificationFailure,
  SecurityParameterNotSet,
  SignatureNotSet,
  KeyDecryptionError,
  BytesToScalarError,
  SHA3DecryptionFailure,
  SymNonceNotSet,
};

enum class SecParam : int { D224 = 224, D256 = 256, D384 = 384, D512 = 512 };

inline std::optional<SecParam> sec_param_try_from(int v) {  // SecParam::try_from, lib.rs:126-134
  switch (v) {
    case 224: return SecParam::D224;
    case 256: return SecParam::D256;
    case 384: return SecParam::D384;
    case 512: return SecParam::D512;
    default: return std::nullopt;
  }
}

using Bytes = std::vector<uint8_t>;
using AffinePoint = std::array<uint8_t, 112>;  // x || y, 56-byte little-endian each

struct Signature {
  Bytes h;                    // 56 bytes
  std::array<uint8_t, 56> z;  // big-endian, canonical
};

struct Message {
  Bytes msg;
  std::optional<SecParam> d;
  std::optional<Bytes> sym_nonce;
  std::optional<AffinePoint> asym_nonce;
  Bytes digest;
  std::optional<Signature> sig;
  explicit Message(Bytes data = {}) : msg(std::move(data)) {}
};

struct KeyPair {
  std::string owner;
  AffinePoint pub_key;
  Bytes priv_key;  // the password, as in the reference
  std::string date_created;
};

struct GpuError : std::runtime_error {
  int status;
  GpuError(int s, const char* what) : std::runtime_error(what), status(s) {}
};

namespace gpu {

namespace detail {
template <class GetBytes, class Items>
inline void pack(const Items& items, GetBytes get, Bytes& data, std::vector<uint64_t>& off) {
  off.assign(items.size() + 1, 0);
  size_t total = 0;
  for (size_t i = 0; i < items.size(); i++) {
    total += get(items[i]).size();
    off[i + 1] = total;
  }
  data.resize(total ? total : 1);
  size_t p = 0;
  for (const auto& it : items) {
    const Bytes& b = get(it);
    std::copy(b.begin(), b.end(), data.begin() + p);
    p += b.size();
  }
}
}  // namespace detail

// A public key prepared on every device of one Engine (Engine::prepare): the comb table of V that the verify /
// key_encrypt overloads taking it use instead of the variable-base ladder.  Reuse it across calls; destroy it before
// the Engine.
class PreparedPublicKey {
 public:
  PreparedPublicKey(PreparedPublicKey&& o) noexcept : key_(o.key_) { o.key_ = nullptr; }
  PreparedPublicKey& operator=(PreparedPublicKey&& o) noexcept {
    if (this != &o) {
      capy_ed448_pub_free(key_);
      key_ = o.key_;
      o.key_ = nullptr;
    }
    return *this;
  }
  PreparedPublicKey(const PreparedPublicKey&) = delete;
  PreparedPublicKey& operator=(const PreparedPublicKey&) = delete;
  ~PreparedPublicKey() { capy_ed448_pub_free(key_); }
  // false when V has a torsion component: the prepared calls then run the generic pipelines (same results)
  bool uses_comb() const { return capy_ed448_pub_uses_comb(key_) == 1; }
  const capy_ed448_pub* raw() const { return key_; }

 private:
  friend class Engine;
  explicit PreparedPublicKey(capy_ed448_pub* k) : key_(k) {}
  capy_ed448_pub* key_ = nullptr;
};

// A batch of resumable SHA3-d or KMACXOF streams (Engine::sha3_hasher / Engine::kmac_xof_hasher): update() appends one
// piece per stream, final() returns what compute_sha3_hash / kmac_xof return for the concatenated pieces.  Destroy it
// before the Engine.
class Hasher {
 public:
  Hasher(Hasher&& o) noexcept : ctx_(o.ctx_), h_(o.h_), n_(o.n_), d_bits_(o.d_bits_), sign_(o.sign_) { o.h_ = nullptr; }
  Hasher& operator=(Hasher&& o) noexcept {
    if (this != &o) {
      capy_hasher_free(h_);
      ctx_ = o.ctx_;
      h_ = o.h_;
      n_ = o.n_;
      d_bits_ = o.d_bits_;
      sign_ = o.sign_;
      o.h_ = nullptr;
    }
    return *this;
  }
  Hasher(const Hasher&) = delete;
  Hasher& operator=(const Hasher&) = delete;
  ~Hasher() { capy_hasher_free(h_); }

  // pieces[i] is appended to stream i
  void update(const std::vector<Bytes>& pieces) {
    if (pieces.size() != n_) throw GpuError(CAPY_ERR_BAD_ARG, "Hasher::update: one piece per stream");
    Bytes data;
    std::vector<uint64_t> off;
    detail::pack(pieces, [](const Bytes& b) -> const Bytes& { return b; }, data, off);
    check(capy_hasher_update(ctx_, h_, data.data(), off.data()));
  }
  // SHA3-d: out_bits = d_bits (0 = d_bits); KMACXOF: out_bits per stream
  std::vector<Bytes> final(uint64_t out_bits = 0) {
    if (out_bits == 0) out_bits = (uint64_t)d_bits_;
    const size_t ob = (size_t)(out_bits / 8);
    Bytes out(n_ * ob + 1);
    check(capy_hasher_final(ctx_, h_, out_bits, nullptr, out.data()));
    std::vector<Bytes> res(n_);
    for (size_t i = 0; i < n_; i++) res[i].assign(out.begin() + i * ob, out.begin() + (i + 1) * ob);
    return res;
  }

  // SHA3-d and KMACXOF streams: the blob of capy_hasher_export, for Engine::import_hasher in this or another Engine (a
  // KMACXOF blob is as secret as its keys)
  Bytes export_blob() {
    uint64_t bytes = 0;
    check(capy_hasher_export_size(h_, &bytes));
    Bytes blob(bytes);
    check(capy_hasher_export(ctx_, h_, blob.data(), bytes));
    return blob;
  }
  // a new hasher on the same Engine: stream j starts as a copy of stream src[j] of this one, which is unchanged (blocking)
  Hasher fork(const std::vector<uint64_t>& src) {
    capy_hasher* f = nullptr;
    check(capy_hasher_fork(ctx_, h_, src.data(), src.size(), &f));
    return Hasher(ctx_, f, src.size(), d_bits_);
  }

  // encryption streams (Engine::sha3_encrypt_stream / key_encrypt_stream): the ciphertext of pieces[i] for every stream;
  // final(512) (sponge AE) or final(448) (key_encrypt) then returns the tags
  std::vector<Bytes> encrypt_update(const std::vector<Bytes>& pieces) {
    if (pieces.size() != n_) throw GpuError(CAPY_ERR_BAD_ARG, "Hasher::encrypt_update: one piece per stream");
    Bytes data;
    std::vector<uint64_t> off;
    detail::pack(pieces, [](const Bytes& b) -> const Bytes& { return b; }, data, off);
    Bytes ct(data.size());
    check(capy_hasher_encrypt_update(ctx_, h_, data.data(), off.data(), ct.data()));
    std::vector<Bytes> res(n_);
    for (size_t i = 0; i < n_; i++) res[i].assign(ct.begin() + off[i], ct.begin() + off[i + 1]);
    return res;
  }

  // verification streams (Engine::verify_stream): ok per stream; *bad_point = a key was off the curve
  Bytes verify_final(bool* bad_point = nullptr) {
    Bytes ok(n_ + 1);
    const int rc = capy_hasher_verify_final(ctx_, h_, ok.data());
    if (rc != CAPY_ERR_BAD_POINT) check(rc);
    if (bad_point) *bad_point = rc == CAPY_ERR_BAD_POINT;
    ok.resize(n_);
    return ok;
  }

  // sign and decryption streams (Engine::sign_stream / sha3_decrypt_stream / key_decrypt_stream): the end of pass 1.
  // Decryption: the verdict per stream; *bad_point = a Z was off the curve.  Sign: an empty result.
  Bytes next_pass(bool* bad_point = nullptr) {
    Bytes ok(n_ + 1);
    const int rc = capy_hasher_next_pass(ctx_, h_, sign_ ? nullptr : ok.data());
    if (rc != CAPY_ERR_BAD_POINT) check(rc);
    if (bad_point) *bad_point = rc == CAPY_ERR_BAD_POINT;
    ok.resize(sign_ ? 0 : n_);
    return ok;
  }
  // decryption pass 2: the plaintext of pieces[i] (the ciphertext where the verdict was 0)
  std::vector<Bytes> decrypt_update(const std::vector<Bytes>& pieces) {
    if (pieces.size() != n_) throw GpuError(CAPY_ERR_BAD_ARG, "Hasher::decrypt_update: one piece per stream");
    Bytes data;
    std::vector<uint64_t> off;
    detail::pack(pieces, [](const Bytes& b) -> const Bytes& { return b; }, data, off);
    check(capy_hasher_decrypt_update(ctx_, h_, data.data(), off.data(), data.data()));
    std::vector<Bytes> res(n_);
    for (size_t i = 0; i < n_; i++) res[i].assign(data.begin() + off[i], data.begin() + off[i + 1]);
    return res;
  }
  Bytes decrypt_final(bool* bad_point = nullptr) {
    Bytes ok(n_ + 1);
    const int rc = capy_hasher_decrypt_final(ctx_, h_, ok.data());
    if (rc != CAPY_ERR_BAD_POINT) check(rc);
    if (bad_point) *bad_point = rc == CAPY_ERR_BAD_POINT;
    ok.resize(n_);
    return ok;
  }
  // the signatures; ok[i] = 0 where pass 2 carried other bytes than pass 1 (then sigs[i] is all zero bytes)
  std::vector<Signature> sign_final(Bytes& ok) {
    Bytes h(n_ * 56 + 1), z(n_ * 56 + 1);
    ok.assign(n_ + 1, 0);
    check(capy_hasher_sign_final(ctx_, h_, h.data(), z.data(), ok.data()));
    ok.resize(n_);
    std::vector<Signature> res(n_);
    for (size_t i = 0; i < n_; i++) {
      res[i].h.assign(h.begin() + 56 * i, h.begin() + 56 * (i + 1));
      std::copy(z.begin() + 56 * i, z.begin() + 56 * (i + 1), res[i].z.begin());
    }
    return res;
  }

 private:
  friend class Engine;
  Hasher(capy_ctx* ctx, capy_hasher* h, size_t n, int d_bits) : ctx_(ctx), h_(h), n_(n), d_bits_(d_bits) {}
  void check(int rc) {
    if (rc != CAPY_OK) throw GpuError(rc, rc == CAPY_ERR_CUDA ? capy_last_cuda_error(ctx_) : capy_strerror(rc));
  }
  capy_ctx* ctx_ = nullptr;
  capy_hasher* h_ = nullptr;
  size_t n_ = 0;
  int d_bits_ = 0;
  bool sign_ = false;  // a sign stream (Engine::sign_stream): next_pass passes no ok
};

class Engine {
 public:
  explicit Engine(const std::vector<int>& devices = {}) {
    int rc = capy_gpu_init(devices.empty() ? nullptr : devices.data(), (int)devices.size(), &ctx_);
    if (rc != CAPY_OK) throw GpuError(rc, capy_strerror(rc));
  }
  ~Engine() { capy_gpu_destroy(ctx_); }
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;

  // SpongeHashable::compute_sha3_hash for every message (sets .digest)
  std::optional<OperationError> compute_sha3_hash(std::vector<Message>& msgs, int d_bits) {
    if (!sec_param_try_from(d_bits)) return OperationError::UnsupportedSecurityParameter;
    Bytes data;
    std::vector<uint64_t> off;
    detail::pack(msgs, [](const Message& m) -> const Bytes& { return m.msg; }, data, off);
    Bytes out(msgs.size() * (size_t)(d_bits / 8));
    check(capy_sha3_batch(ctx_, d_bits, data.data(), off.data(), msgs.size(), out.data(), 0));
    for (size_t i = 0; i < msgs.size(); i++)
      msgs[i].digest.assign(out.begin() + i * (d_bits / 8), out.begin() + (i + 1) * (d_bits / 8));
    return std::nullopt;
  }

  // SpongeHashable::compute_tagged_hash: digest = kmac_xof(pw, msg, d, s, d)
  std::optional<OperationError> compute_tagged_hash(std::vector<Message>& msgs, const std::vector<Bytes>& pws,
                                                    const std::string& s, int d_bits) {
    if (!sec_param_try_from(d_bits)) return OperationError::UnsupportedSecurityParameter;
    auto out = kmac_xof(pws, msgs, (uint64_t)d_bits, s, d_bits);
    for (size_t i = 0; i < msgs.size(); i++) msgs[i].digest = std::move(out[i]);
    return std::nullopt;
  }

  // pub fn kmac_xof, one (key, message) pair per item
  std::vector<Bytes> kmac_xof(const std::vector<Bytes>& keys, const std::vector<Message>& msgs, uint64_t l_bits,
                              const std::string& s, int d_bits) {
    Bytes kd, xd;
    std::vector<uint64_t> ko, xo;
    detail::pack(keys, [](const Bytes& b) -> const Bytes& { return b; }, kd, ko);
    detail::pack(msgs, [](const Message& m) -> const Bytes& { return m.msg; }, xd, xo);
    const size_t ob = (size_t)(l_bits / 8);
    Bytes out(msgs.size() * ob + 1);
    check(capy_kmac_xof_batch(ctx_, d_bits, kd.data(), ko.data(), xd.data(), xo.data(), msgs.size(),
                              reinterpret_cast<const uint8_t*>(s.data()), (uint32_t)s.size(), l_bits, nullptr, out.data()));
    std::vector<Bytes> res(msgs.size());
    for (size_t i = 0; i < msgs.size(); i++) res[i].assign(out.begin() + i * ob, out.begin() + (i + 1) * ob);
    return res;
  }

  // n SHA3-d streams fed in pieces (blocking)
  Hasher sha3_hasher(size_t n, int d_bits) {
    capy_hasher* h = nullptr;
    check(capy_sha3_hasher_new(ctx_, d_bits, n, &h));
    return Hasher(ctx_, h, n, d_bits);
  }

  // one KMACXOF stream per key, customisation string s (blocking); d_bits = 224 is refused (CAPY_ERR_BAD_ARG)
  Hasher kmac_xof_hasher(const std::vector<Bytes>& keys, const std::string& s, int d_bits) {
    Bytes kd;
    std::vector<uint64_t> ko;
    detail::pack(keys, [](const Bytes& b) -> const Bytes& { return b; }, kd, ko);
    capy_hasher* h = nullptr;
    check(capy_kmac_xof_hasher_new(ctx_, d_bits, kd.data(), ko.data(), keys.size(),
                                   reinterpret_cast<const uint8_t*>(s.data()), (uint32_t)s.size(), &h));
    return Hasher(ctx_, h, keys.size(), d_bits);
  }

  // the streams of a blob from Hasher::export_blob, dealt over this Engine's devices (blocking)
  Hasher import_hasher(const Bytes& blob) {
    int d_bits = 0;
    uint64_t n = 0;
    check(capy_hasher_blob_info(blob.data(), blob.size(), nullptr, &d_bits, &n));
    capy_hasher* h = nullptr;
    check(capy_hasher_import(ctx_, blob.data(), blob.size(), &h));
    return Hasher(ctx_, h, (size_t)n, d_bits);
  }

  // sha3_encrypt of plaintexts fed in pieces (Hasher::encrypt_update, then final(512) for the tags): one stream per
  // password, nonces[i] its 512-byte z (blocking); d_bits = 224 is refused (CAPY_ERR_BAD_ARG)
  Hasher sha3_encrypt_stream(const std::vector<Bytes>& pws, const std::vector<Bytes>& nonces, int d_bits) {
    Bytes pd, zs;
    std::vector<uint64_t> po;
    detail::pack(pws, [](const Bytes& b) -> const Bytes& { return b; }, pd, po);
    for (const Bytes& z : nonces) {
      if (z.size() != 512) throw GpuError(CAPY_ERR_BAD_ARG, "sha3_encrypt_stream: 512-byte nonces");
      zs.insert(zs.end(), z.begin(), z.end());
    }
    if (nonces.size() != pws.size()) throw GpuError(CAPY_ERR_BAD_ARG, "sha3_encrypt_stream: one nonce per password");
    zs.push_back(0);
    capy_hasher* h = nullptr;
    check(capy_sponge_encrypt_stream_new(ctx_, d_bits, CAPY_AE_SHA3, pd.data(), po.data(), zs.data(), 512, pws.size(), &h));
    return Hasher(ctx_, h, pws.size(), d_bits);
  }

  // key_encrypt of plaintexts fed in pieces to one prepared key (then final(448) for the tags); z[i] <- Z_i (blocking)
  Hasher key_encrypt_stream(const PreparedPublicKey& key, const std::vector<std::array<uint8_t, 56>>& k_rand, int d_bits,
                            std::vector<AffinePoint>& z) {
    const size_t n = k_rand.size();
    Bytes ks(n * 56 + 1), zb(n * 112 + 1);
    for (size_t i = 0; i < n; i++) std::copy(k_rand[i].begin(), k_rand[i].end(), ks.begin() + 56 * i);
    capy_hasher* h = nullptr;
    check(capy_ed448_key_encrypt_stream_new(ctx_, d_bits, nullptr, key.raw(), ks.data(), n, zb.data(), &h));
    z.resize(n);
    for (size_t i = 0; i < n; i++) std::copy(zb.begin() + 112 * i, zb.begin() + 112 * (i + 1), z[i].begin());
    return Hasher(ctx_, h, n, d_bits);
  }

  // verify of messages fed in pieces (Hasher::update, then Hasher::verify_final) against one prepared key (blocking)
  Hasher verify_stream(const std::vector<Signature>& sigs, const PreparedPublicKey& key, int d_bits) {
    Bytes h, z;
    for (const Signature& s : sigs) {
      if (s.h.size() != 56) throw GpuError(CAPY_ERR_BAD_ARG, "verify_stream: 56-byte h");
      h.insert(h.end(), s.h.begin(), s.h.end());
      z.insert(z.end(), s.z.begin(), s.z.end());
    }
    h.push_back(0);
    z.push_back(0);
    capy_hasher* hs = nullptr;
    check(capy_ed448_verify_stream_new(ctx_, d_bits, nullptr, key.raw(), h.data(), z.data(), sigs.size(), &hs));
    return Hasher(ctx_, hs, sigs.size(), d_bits);
  }

  // sign of messages fed twice in pieces: update, next_pass, update, sign_final (blocking creation)
  Hasher sign_stream(const std::vector<Bytes>& pws, int d_bits) {
    Bytes pd;
    std::vector<uint64_t> po;
    detail::pack(pws, [](const Bytes& b) -> const Bytes& { return b; }, pd, po);
    capy_hasher* h = nullptr;
    check(capy_ed448_sign_stream_new(ctx_, d_bits, pd.data(), po.data(), pws.size(), &h));
    Hasher r(ctx_, h, pws.size(), d_bits);
    r.sign_ = true;
    return r;
  }

  // sha3_decrypt of ciphertexts fed twice: update, next_pass, decrypt_update, decrypt_final (512-byte nonces)
  Hasher sha3_decrypt_stream(const std::vector<Bytes>& pws, const std::vector<Bytes>& nonces, const std::vector<Bytes>& tags,
                             int d_bits) {
    if (nonces.size() != pws.size() || tags.size() != pws.size())
      throw GpuError(CAPY_ERR_BAD_ARG, "sha3_decrypt_stream: one nonce and one tag per password");
    Bytes pd, zs, ts;
    std::vector<uint64_t> po;
    detail::pack(pws, [](const Bytes& b) -> const Bytes& { return b; }, pd, po);
    for (size_t i = 0; i < pws.size(); i++) {
      if (nonces[i].size() != 512 || tags[i].size() != 64)
        throw GpuError(CAPY_ERR_BAD_ARG, "sha3_decrypt_stream: 512-byte nonces and 64-byte tags");
      zs.insert(zs.end(), nonces[i].begin(), nonces[i].end());
      ts.insert(ts.end(), tags[i].begin(), tags[i].end());
    }
    zs.push_back(0);
    ts.push_back(0);
    capy_hasher* h = nullptr;
    check(capy_sponge_decrypt_stream_new(ctx_, d_bits, CAPY_AE_SHA3, pd.data(), po.data(), zs.data(), 512, ts.data(),
                                         pws.size(), &h));
    return Hasher(ctx_, h, pws.size(), d_bits);
  }

  // key_decrypt of ciphertexts fed twice (z[i] = Z_i, 56-byte tags)
  Hasher key_decrypt_stream(const std::vector<Bytes>& pws, const std::vector<AffinePoint>& z, const std::vector<Bytes>& tags,
                            int d_bits) {
    if (z.size() != pws.size() || tags.size() != pws.size())
      throw GpuError(CAPY_ERR_BAD_ARG, "key_decrypt_stream: one Z and one tag per password");
    Bytes pd, zs, ts;
    std::vector<uint64_t> po;
    detail::pack(pws, [](const Bytes& b) -> const Bytes& { return b; }, pd, po);
    for (size_t i = 0; i < pws.size(); i++) {
      if (tags[i].size() != 56) throw GpuError(CAPY_ERR_BAD_ARG, "key_decrypt_stream: 56-byte tags");
      zs.insert(zs.end(), z[i].begin(), z[i].end());
      ts.insert(ts.end(), tags[i].begin(), tags[i].end());
    }
    zs.push_back(0);
    ts.push_back(0);
    capy_hasher* h = nullptr;
    check(capy_ed448_key_decrypt_stream_new(ctx_, d_bits, pd.data(), po.data(), zs.data(), ts.data(), pws.size(), &h));
    return Hasher(ctx_, h, pws.size(), d_bits);
  }

  // KeyPair::new for every password
  std::vector<KeyPair> new_keypairs(const std::vector<Bytes>& pws, const std::string& owner, int d_bits) {
    Bytes pd;
    std::vector<uint64_t> po;
    detail::pack(pws, [](const Bytes& b) -> const Bytes& { return b; }, pd, po);
    Bytes out(pws.size() * 112 + 1);
    check(capy_ed448_keygen_batch(ctx_, d_bits, pd.data(), po.data(), pws.size(), out.data()));
    std::vector<KeyPair> kp(pws.size());
    for (size_t i = 0; i < pws.size(); i++) {
      kp[i].owner = owner;
      std::copy(out.begin() + 112 * i, out.begin() + 112 * (i + 1), kp[i].pub_key.begin());
      kp[i].priv_key = pws[i];
    }
    return kp;
  }

  // Signable::sign: message i is signed under keys[i]
  void sign(std::vector<Message>& msgs, const std::vector<KeyPair>& keys, int d_bits) {
    Bytes pd, md;
    std::vector<uint64_t> po, mo;
    detail::pack(keys, [](const KeyPair& k) -> const Bytes& { return k.priv_key; }, pd, po);
    detail::pack(msgs, [](const Message& m) -> const Bytes& { return m.msg; }, md, mo);
    Bytes h(msgs.size() * 56 + 1), z(msgs.size() * 56 + 1);
    check(capy_ed448_sign_batch(ctx_, d_bits, pd.data(), po.data(), md.data(), mo.data(), msgs.size(), h.data(), z.data()));
    for (size_t i = 0; i < msgs.size(); i++) {
      Signature s;
      s.h.assign(h.begin() + 56 * i, h.begin() + 56 * (i + 1));
      std::copy(z.begin() + 56 * i, z.begin() + 56 * (i + 1), s.z.begin());
      msgs[i].sig = std::move(s);
      msgs[i].d = *sec_param_try_from(d_bits);
    }
  }

  // Signable::verify: result[i] is empty for Ok(()), else the reference's error
  std::vector<std::optional<OperationError>> verify(const std::vector<Message>& msgs, const std::vector<AffinePoint>& pubs) {
    std::vector<std::optional<OperationError>> res(msgs.size());
    for (int d_bits : {224, 256, 384, 512}) {
      std::vector<size_t> idx;
      for (size_t i = 0; i < msgs.size(); i++) {
        if (!msgs[i].sig) res[i] = OperationError::SignatureNotSet;
        else if (!msgs[i].d) res[i] = OperationError::SecurityParameterNotSet;
        else if ((int)*msgs[i].d == d_bits) idx.push_back(i);
      }
      if (idx.empty()) continue;
      Bytes md, pub, h, z;
      std::vector<uint64_t> mo(1, 0);
      for (size_t i : idx) {
        md.insert(md.end(), msgs[i].msg.begin(), msgs[i].msg.end());
        mo.push_back(md.size());
        pub.insert(pub.end(), pubs[i].begin(), pubs[i].end());
        h.insert(h.end(), msgs[i].sig->h.begin(), msgs[i].sig->h.end());
        z.insert(z.end(), msgs[i].sig->z.begin(), msgs[i].sig->z.end());
      }
      if (md.empty()) md.push_back(0);
      Bytes ok(idx.size());
      int rc = capy_ed448_verify_batch(ctx_, d_bits, pub.data(), md.data(), mo.data(), h.data(), z.data(), idx.size(), ok.data());
      if (rc != CAPY_OK && rc != CAPY_ERR_BAD_POINT) check(rc);
      for (size_t k = 0; k < idx.size(); k++)
        if (!ok[k]) res[idx[k]] = OperationError::SignatureVerificationFailure;
    }
    return res;
  }

  // prepares V for many verify / key_encrypt calls (blocking); GpuError(CAPY_ERR_BAD_POINT) when V is off the curve
  PreparedPublicKey prepare(const AffinePoint& pub) {
    capy_ed448_pub* k = nullptr;
    check(capy_ed448_pub_prepare(ctx_, pub.data(), &k));
    return PreparedPublicKey(k);
  }

  // Signable::verify of every message against one signer: result[i] as verify() gives it with pubs[i] = the key
  std::vector<std::optional<OperationError>> verify(const std::vector<Message>& msgs, const PreparedPublicKey& key) {
    std::vector<std::optional<OperationError>> res(msgs.size());
    for (int d_bits : {224, 256, 384, 512}) {
      std::vector<size_t> idx;
      for (size_t i = 0; i < msgs.size(); i++) {
        if (!msgs[i].sig) res[i] = OperationError::SignatureNotSet;
        else if (!msgs[i].d) res[i] = OperationError::SecurityParameterNotSet;
        else if ((int)*msgs[i].d == d_bits) {
          if (msgs[i].sig->h.size() != 56) res[i] = OperationError::SignatureVerificationFailure;
          else idx.push_back(i);
        }
      }
      if (idx.empty()) continue;
      Bytes md, h, z;
      std::vector<uint64_t> mo(1, 0);
      for (size_t i : idx) {
        md.insert(md.end(), msgs[i].msg.begin(), msgs[i].msg.end());
        mo.push_back(md.size());
        h.insert(h.end(), msgs[i].sig->h.begin(), msgs[i].sig->h.end());
        z.insert(z.end(), msgs[i].sig->z.begin(), msgs[i].sig->z.end());
      }
      if (md.empty()) md.push_back(0);
      Bytes ok(idx.size());
      check(capy_ed448_verify_prepared_batch(ctx_, d_bits, key.raw(), md.data(), mo.data(), h.data(), z.data(), idx.size(),
                                             ok.data()));
      for (size_t k = 0; k < idx.size(); k++)
        if (!ok[k]) res[idx[k]] = OperationError::SignatureVerificationFailure;
    }
    return res;
  }

  // KeyEncryptable::key_encrypt of every message to one recipient (as key_encrypt() with pubs[i] = the key)
  std::optional<OperationError> key_encrypt(std::vector<Message>& msgs, const PreparedPublicKey& key, int d_bits,
                                            const std::vector<std::array<uint8_t, 56>>* k_rand = nullptr) {
    if (!sec_param_try_from(d_bits)) return OperationError::UnsupportedSecurityParameter;
    const size_t n = msgs.size();
    Bytes md, ks(n * 56 + 1);
    std::vector<uint64_t> mo;
    detail::pack(msgs, [](const Message& m) -> const Bytes& { return m.msg; }, md, mo);
    std::random_device rd;
    for (size_t i = 0; i < n; i++)
      for (size_t k = 0; k < 56; k++) ks[56 * i + k] = k_rand ? (*k_rand)[i][k] : (uint8_t)rd();
    Bytes ct(md.size()), tag(n * 56 + 1), z(n * 112 + 1);
    check(capy_ed448_key_encrypt_prepared_batch(ctx_, d_bits, key.raw(), ks.data(), md.data(), mo.data(), n, ct.data(),
                                                tag.data(), z.data()));
    for (size_t i = 0; i < n; i++) {
      msgs[i].msg.assign(ct.begin() + mo[i], ct.begin() + mo[i + 1]);
      msgs[i].digest.assign(tag.begin() + 56 * i, tag.begin() + 56 * (i + 1));
      AffinePoint zp;
      std::copy(z.begin() + 112 * i, z.begin() + 112 * (i + 1), zp.begin());
      msgs[i].asym_nonce = zp;
      msgs[i].d = *sec_param_try_from(d_bits);
    }
    return std::nullopt;
  }

  // SpongeEncryptable::sha3_encrypt (sha3/encryptable.rs:29-45): msg <- ciphertext, digest <- tag, sym_nonce <- z.
  // z = 512 random bytes per message (:31) drawn on the host unless `nonces` is given.
  std::optional<OperationError> sha3_encrypt(std::vector<Message>& msgs, const std::vector<Bytes>& pws, int d_bits,
                                             const std::vector<Bytes>* nonces = nullptr) {
    if (!sec_param_try_from(d_bits)) return OperationError::UnsupportedSecurityParameter;
    const size_t n = msgs.size();
    Bytes pd, md, zs(n * 512 + 1);
    std::vector<uint64_t> po, mo;
    detail::pack(pws, [](const Bytes& b) -> const Bytes& { return b; }, pd, po);
    detail::pack(msgs, [](const Message& m) -> const Bytes& { return m.msg; }, md, mo);
    std::random_device rd;
    for (size_t i = 0; i < n; i++)
      for (size_t k = 0; k < 512; k++) zs[512 * i + k] = nonces ? (*nonces)[i][k] : (uint8_t)rd();
    Bytes ct(md.size()), tag(n * 64 + 1);
    check(capy_sponge_encrypt_batch(ctx_, d_bits, CAPY_AE_SHA3, pd.data(), po.data(), zs.data(), 512, md.data(), mo.data(), n,
                                    ct.data(), tag.data()));
    for (size_t i = 0; i < n; i++) {
      msgs[i].msg.assign(ct.begin() + mo[i], ct.begin() + mo[i + 1]);
      msgs[i].digest.assign(tag.begin() + 64 * i, tag.begin() + 64 * (i + 1));
      msgs[i].sym_nonce = Bytes(zs.begin() + 512 * i, zs.begin() + 512 * (i + 1));
      msgs[i].d = *sec_param_try_from(d_bits);
    }
    return std::nullopt;
  }

  // SpongeEncryptable::sha3_decrypt (:58-83): empty for Ok(()); on failure msg keeps the ciphertext
  std::vector<std::optional<OperationError>> sha3_decrypt(std::vector<Message>& msgs, const std::vector<Bytes>& pws) {
    std::vector<std::optional<OperationError>> res(msgs.size());
    for (int d_bits : {224, 256, 384, 512}) {
      std::vector<size_t> idx;
      for (size_t i = 0; i < msgs.size(); i++) {
        if (!msgs[i].d) res[i] = OperationError::SecurityParameterNotSet;
        else if (!msgs[i].sym_nonce) res[i] = OperationError::SymNonceNotSet;
        else if ((int)*msgs[i].d == d_bits) {
          if (msgs[i].sym_nonce->size() != 512 || msgs[i].digest.size() != 64) res[i] = OperationError::SHA3DecryptionFailure;
          else idx.push_back(i);
        }
      }
      if (idx.empty()) continue;
      Bytes pd, cd, zs, tags;
      std::vector<uint64_t> po(1, 0), co(1, 0);
      for (size_t i : idx) {
        pd.insert(pd.end(), pws[i].begin(), pws[i].end());
        po.push_back(pd.size());
        cd.insert(cd.end(), msgs[i].msg.begin(), msgs[i].msg.end());
        co.push_back(cd.size());
        zs.insert(zs.end(), msgs[i].sym_nonce->begin(), msgs[i].sym_nonce->end());
        tags.insert(tags.end(), msgs[i].digest.begin(), msgs[i].digest.end());
      }
      if (pd.empty()) pd.push_back(0);
      if (cd.empty()) cd.push_back(0);
      Bytes out(cd.size()), ok(idx.size());
      check(capy_sponge_decrypt_batch(ctx_, d_bits, CAPY_AE_SHA3, pd.data(), po.data(), zs.data(), 512, cd.data(), co.data(),
                                      tags.data(), idx.size(), out.data(), ok.data()));
      for (size_t k = 0; k < idx.size(); k++) {
        if (ok[k]) msgs[idx[k]].msg.assign(out.begin() + co[k], out.begin() + co[k + 1]);
        else res[idx[k]] = OperationError::SHA3DecryptionFailure;
      }
    }
    return res;
  }

  // KeyEncryptable::key_encrypt (ecc/encryptable.rs:34-50): msg <- ciphertext, digest <- tag, asym_nonce <- Z.
  // k = 56 random bytes per message (:36) drawn on the host unless `k_rand` is given.
  std::optional<OperationError> key_encrypt(std::vector<Message>& msgs, const std::vector<AffinePoint>& pubs, int d_bits,
                                            const std::vector<std::array<uint8_t, 56>>* k_rand = nullptr) {
    if (!sec_param_try_from(d_bits)) return OperationError::UnsupportedSecurityParameter;
    const size_t n = msgs.size();
    Bytes md, pub(n * 112 + 1), ks(n * 56 + 1);
    std::vector<uint64_t> mo;
    detail::pack(msgs, [](const Message& m) -> const Bytes& { return m.msg; }, md, mo);
    std::random_device rd;
    for (size_t i = 0; i < n; i++) {
      std::copy(pubs[i].begin(), pubs[i].end(), pub.begin() + 112 * i);
      for (size_t k = 0; k < 56; k++) ks[56 * i + k] = k_rand ? (*k_rand)[i][k] : (uint8_t)rd();
    }
    Bytes ct(md.size()), tag(n * 56 + 1), z(n * 112 + 1);
    check(capy_ed448_key_encrypt_batch(ctx_, d_bits, pub.data(), ks.data(), md.data(), mo.data(), n, ct.data(), tag.data(),
                                       z.data()));
    for (size_t i = 0; i < n; i++) {
      msgs[i].msg.assign(ct.begin() + mo[i], ct.begin() + mo[i + 1]);
      msgs[i].digest.assign(tag.begin() + 56 * i, tag.begin() + 56 * (i + 1));
      AffinePoint zp;
      std::copy(z.begin() + 112 * i, z.begin() + 112 * (i + 1), zp.begin());
      msgs[i].asym_nonce = zp;
      msgs[i].d = *sec_param_try_from(d_bits);
    }
    return std::nullopt;
  }

  // KeyEncryptable::key_decrypt (:72-94): empty for Ok(()); SymNonceNotSet (sic, :73) when asym_nonce is missing
  std::vector<std::optional<OperationError>> key_decrypt(std::vector<Message>& msgs, const std::vector<Bytes>& pws) {
    std::vector<std::optional<OperationError>> res(msgs.size());
    for (int d_bits : {224, 256, 384, 512}) {
      std::vector<size_t> idx;
      for (size_t i = 0; i < msgs.size(); i++) {
        if (!msgs[i].asym_nonce) res[i] = OperationError::SymNonceNotSet;
        else if (!msgs[i].d) res[i] = OperationError::SecurityParameterNotSet;
        else if ((int)*msgs[i].d == d_bits) {
          if (msgs[i].digest.size() != 56) res[i] = OperationError::KeyDecryptionError;
          else idx.push_back(i);
        }
      }
      if (idx.empty()) continue;
      Bytes pd, cd, zs, tags;
      std::vector<uint64_t> po(1, 0), co(1, 0);
      for (size_t i : idx) {
        pd.insert(pd.end(), pws[i].begin(), pws[i].end());
        po.push_back(pd.size());
        cd.insert(cd.end(), msgs[i].msg.begin(), msgs[i].msg.end());
        co.push_back(cd.size());
        zs.insert(zs.end(), msgs[i].asym_nonce->begin(), msgs[i].asym_nonce->end());
        tags.insert(tags.end(), msgs[i].digest.begin(), msgs[i].digest.end());
      }
      if (pd.empty()) pd.push_back(0);
      if (cd.empty()) cd.push_back(0);
      Bytes out(cd.size()), ok(idx.size());
      int rc = capy_ed448_key_decrypt_batch(ctx_, d_bits, pd.data(), po.data(), zs.data(), cd.data(), co.data(), tags.data(),
                                            idx.size(), out.data(), ok.data());
      if (rc != CAPY_OK && rc != CAPY_ERR_BAD_POINT) check(rc);
      for (size_t k = 0; k < idx.size(); k++) {
        if (ok[k]) msgs[idx[k]].msg.assign(out.begin() + co[k], out.begin() + co[k + 1]);
        else res[idx[k]] = OperationError::KeyDecryptionError;
      }
    }
    return res;
  }

  capy_ctx* raw() { return ctx_; }

 private:
  void check(int rc) {
    if (rc != CAPY_OK) throw GpuError(rc, rc == CAPY_ERR_CUDA ? capy_last_cuda_error(ctx_) : capy_strerror(rc));
  }
  capy_ctx* ctx_ = nullptr;
};

}  // namespace gpu
}  // namespace capycrypt
