// tests/host/two_pass_mirror_check.cpp -- the sign and decryption streams of the C++ host mirror
// (capycrypt_b200/host/capycrypt_gpu.hpp): messages fed twice in pieces through Engine::sign_stream,
// Engine::sha3_decrypt_stream and Engine::key_decrypt_stream give what sign, sha3_decrypt and key_decrypt give for the
// whole messages, and a pass 2 over other bytes fails.  Needs a GPU; compiled and run by tests/test_two_pass_streams_gpu.py.
#include <cstdio>
#include "../../capycrypt_b200/host/capycrypt_gpu.hpp"
using namespace capycrypt;

#define EXPECT(c) do { if (!(c)) { printf("FAIL line %d: %s\n", __LINE__, #c); return 1; } } while (0)

static std::vector<Bytes> cut(const std::vector<Bytes>& whole, size_t k, size_t updates) {
  std::vector<Bytes> p(whole.size());
  for (size_t i = 0; i < whole.size(); i++) {
    const size_t a = whole[i].size() * k / updates, b = whole[i].size() * (k + 1) / updates;
    p[i].assign(whole[i].begin() + a, whole[i].begin() + b);
  }
  return p;
}

int main() {
  gpu::Engine eng;
  const size_t n = 3;
  std::vector<Bytes> msgs(n);
  for (size_t i = 0; i < n; i++)
    for (size_t b = 0; b < 97 * i + 140; b++) msgs[i].push_back((uint8_t)(i * 13 + b));
  const std::vector<Bytes> pws = {Bytes{1, 2, 3}, Bytes(), Bytes(40, 0x07)};
  std::vector<Bytes> nonces(n);
  for (size_t i = 0; i < n; i++)
    for (size_t b = 0; b < 512; b++) nonces[i].push_back((uint8_t)(i + 3 * b));
  std::vector<std::array<uint8_t, 56>> k_rand(n);
  for (size_t i = 0; i < n; i++)
    for (size_t b = 0; b < 56; b++) k_rand[i][b] = (uint8_t)(5 * i + b);
  for (int d : {256, 384, 512}) {
    std::vector<Message> ref;
    for (const Bytes& m : msgs) ref.emplace_back(m);
    // sign: pass 1 in three pieces, pass 2 in two; item 2 differs in pass 2
    auto kps = eng.new_keypairs(pws, "mirror", d);
    eng.sign(ref, kps, d);
    gpu::Hasher ss = eng.sign_stream(pws, d);
    for (size_t k = 0; k < 3; k++) ss.update(cut(msgs, k, 3));
    ss.next_pass();
    std::vector<Bytes> other = msgs;
    other[2][5] ^= 1;
    for (size_t k = 0; k < 2; k++) ss.update(cut(other, k, 2));
    Bytes ok;
    auto sigs = ss.sign_final(ok);
    EXPECT(ok[0] == 1 && ok[1] == 1 && ok[2] == 0);
    for (size_t i = 0; i < 2; i++) EXPECT(sigs[i].h == ref[i].sig->h && sigs[i].z == ref[i].sig->z);
    EXPECT(sigs[2].h == Bytes(56, 0) && sigs[2].z == (std::array<uint8_t, 56>{}));
    // sha3_decrypt
    ref.clear();
    for (const Bytes& m : msgs) ref.emplace_back(m);
    EXPECT(!eng.sha3_encrypt(ref, pws, d, &nonces));
    std::vector<Bytes> cts, tags;
    for (const Message& m : ref) {
      cts.push_back(m.msg);
      tags.push_back(m.digest);
    }
    gpu::Hasher ds = eng.sha3_decrypt_stream(pws, nonces, tags, d);
    for (size_t k = 0; k < 4; k++) ds.update(cut(cts, k, 4));
    Bytes verdict = ds.next_pass();
    EXPECT(verdict == Bytes(n, 1));
    std::vector<Bytes> pt(n);
    for (size_t k = 0; k < 2; k++) {
      auto p = ds.decrypt_update(cut(cts, k, 2));
      for (size_t i = 0; i < n; i++) pt[i].insert(pt[i].end(), p[i].begin(), p[i].end());
    }
    EXPECT(ds.decrypt_final() == Bytes(n, 1) && pt == msgs);
    // key_decrypt
    ref.clear();
    for (const Bytes& m : msgs) ref.emplace_back(m);
    gpu::PreparedPublicKey key = eng.prepare(kps[0].pub_key);
    EXPECT(!eng.key_encrypt(ref, key, d, &k_rand));
    std::vector<AffinePoint> z;
    cts.clear();
    tags.clear();
    for (const Message& m : ref) {
      cts.push_back(m.msg);
      tags.push_back(m.digest);
      z.push_back(*m.asym_nonce);
    }
    gpu::Hasher kd = eng.key_decrypt_stream(std::vector<Bytes>(n, pws[0]), z, tags, d);
    kd.update(cts);
    bool bad = true;
    EXPECT(kd.next_pass(&bad) == Bytes(n, 1) && !bad);
    EXPECT(kd.decrypt_update(cts) == msgs && kd.decrypt_final() == Bytes(n, 1));
  }
  bool refused = false;
  try {
    eng.sign_stream(pws, 224);
  } catch (const GpuError& e) {
    refused = e.status == CAPY_ERR_BAD_ARG;
  }
  EXPECT(refused);
  printf("OK\n");
  return 0;
}
