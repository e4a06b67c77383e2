// tests/host/streams_mirror_check.cpp -- the encryption and verification streams of the C++ host mirror
// (capycrypt_b200/host/capycrypt_gpu.hpp): plaintexts and messages fed in pieces through Engine::sha3_encrypt_stream,
// Engine::key_encrypt_stream and Engine::verify_stream give what sha3_encrypt, key_encrypt and verify give for the whole
// messages.  Needs a GPU; compiled and run by tests/test_streams_gpu.py.
#include <cstdio>
#include "../../capycrypt_b200/host/capycrypt_gpu.hpp"
using namespace capycrypt;

#define EXPECT(c) do { if (!(c)) { printf("FAIL line %d: %s\n", __LINE__, #c); return 1; } } while (0)

int main() {
  gpu::Engine eng;
  // three streams, four updates: item i's piece k has (37 i + 61 k) % 150 bytes (some empty)
  const size_t n = 3, updates = 4;
  std::vector<Message> whole(n);
  std::vector<std::vector<Bytes>> pieces(updates, std::vector<Bytes>(n));
  for (size_t k = 0; k < updates; k++)
    for (size_t i = 0; i < n; i++) {
      const size_t len = (37 * i + 61 * k) % 150;
      for (size_t b = 0; b < len; b++) pieces[k][i].push_back((uint8_t)(i * 31 + k * 7 + b));
      whole[i].msg.insert(whole[i].msg.end(), pieces[k][i].begin(), pieces[k][i].end());
    }
  const std::vector<Bytes> pws = {Bytes{1, 2, 3}, Bytes(), Bytes(40, 0x07)};
  std::vector<Bytes> nonces(n);
  for (size_t i = 0; i < n; i++)
    for (size_t b = 0; b < 512; b++) nonces[i].push_back((uint8_t)(i + 3 * b));
  std::vector<std::array<uint8_t, 56>> k_rand(n);
  for (size_t i = 0; i < n; i++)
    for (size_t b = 0; b < 56; b++) k_rand[i][b] = (uint8_t)(5 * i + b);
  for (int d : {256, 384, 512}) {
    // sha3_encrypt
    std::vector<Message> ref = whole;
    EXPECT(!eng.sha3_encrypt(ref, pws, d, &nonces));
    gpu::Hasher st = eng.sha3_encrypt_stream(pws, nonces, d);
    std::vector<Bytes> ct(n);
    for (size_t k = 0; k < updates; k++) {
      auto c = st.encrypt_update(pieces[k]);
      for (size_t i = 0; i < n; i++) ct[i].insert(ct[i].end(), c[i].begin(), c[i].end());
    }
    auto tags = st.final(512);
    for (size_t i = 0; i < n; i++) EXPECT(ct[i] == ref[i].msg && tags[i] == ref[i].digest);
    bool refused = false;
    try {
      st.update(pieces[0]);  // an encryption stream takes encrypt_update only
    } catch (const GpuError& e) {
      refused = e.status == CAPY_ERR_BAD_ARG;
    }
    EXPECT(refused);
    // key_encrypt and verify against one prepared key
    auto kp = eng.new_keypairs({Bytes{9, 9, 9}}, "mirror", d);
    gpu::PreparedPublicKey key = eng.prepare(kp[0].pub_key);
    ref = whole;
    EXPECT(!eng.key_encrypt(ref, key, d, &k_rand));
    std::vector<AffinePoint> z;
    gpu::Hasher ke = eng.key_encrypt_stream(key, k_rand, d, z);
    std::vector<Bytes> kct(n);
    for (size_t k = 0; k < updates; k++) {
      auto c = ke.encrypt_update(pieces[k]);
      for (size_t i = 0; i < n; i++) kct[i].insert(kct[i].end(), c[i].begin(), c[i].end());
    }
    auto ktags = ke.final(448);
    for (size_t i = 0; i < n; i++) EXPECT(kct[i] == ref[i].msg && ktags[i] == ref[i].digest && z[i] == *ref[i].asym_nonce);
    std::vector<Message> sm = whole;
    std::vector<KeyPair> signers(n, kp[0]);
    eng.sign(sm, signers, d);
    std::vector<Signature> sigs;
    for (const Message& m : sm) sigs.push_back(*m.sig);
    sigs[1].h[0] ^= 1;
    gpu::Hasher vs = eng.verify_stream(sigs, key, d);
    for (size_t k = 0; k < updates; k++) vs.update(pieces[k]);
    bool bad = true;
    Bytes ok = vs.verify_final(&bad);
    EXPECT(!bad && ok[0] == 1 && ok[1] == 0 && ok[2] == 1);
  }
  bool refused = false;
  try {
    eng.sha3_encrypt_stream(pws, nonces, 224);
  } catch (const GpuError& e) {
    refused = e.status == CAPY_ERR_BAD_ARG;
  }
  EXPECT(refused);
  printf("OK\n");
  return 0;
}
