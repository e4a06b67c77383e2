// tests/host/prepared_mirror_check.cpp -- the prepared-key methods of the C++ host mirror
// (capycrypt_b200/host/capycrypt_gpu.hpp): verify against one signer and key_encrypt to one recipient give what the
// per-message-key methods give.  Needs a GPU; compiled and run by tests/test_ed448_prepared_gpu.py.
#include <cstdio>
#include <cstring>
#include "../../capycrypt_b200/host/capycrypt_gpu.hpp"
using namespace capycrypt;

#define EXPECT(c) do { if (!(c)) { printf("FAIL line %d: %s\n", __LINE__, #c); return 1; } } while (0)

int main() {
  gpu::Engine eng;
  std::vector<Bytes> pws = {Bytes(64, 7)};
  auto keys = eng.new_keypairs(pws, "signer", 512);
  const AffinePoint pub = keys[0].pub_key;
  gpu::PreparedPublicKey key = eng.prepare(pub);
  EXPECT(key.uses_comb());
  // sign five messages with the one key, then tamper with two of them
  std::vector<Message> s;
  for (int i = 0; i < 5; i++) s.emplace_back(Bytes(100 + 37 * i, (uint8_t)i));
  eng.sign(s, std::vector<KeyPair>(s.size(), keys[0]), 512);
  s[1].msg[0] ^= 1;
  s[3].sig->h[5] ^= 1;
  s.emplace_back(Bytes{1, 2, 3});  // not signed
  auto want = eng.verify(s, std::vector<AffinePoint>(s.size(), pub));
  auto got = eng.verify(s, key);
  EXPECT(got == want);
  EXPECT(!got[0] && !got[2] && !got[4]);
  EXPECT(got[1] == OperationError::SignatureVerificationFailure && got[3] == OperationError::SignatureVerificationFailure);
  EXPECT(got[5] == OperationError::SignatureNotSet);
  // key_encrypt to the one recipient: the same bytes as with the key repeated, and key_decrypt opens them
  std::vector<std::array<uint8_t, 56>> k(3);
  for (size_t i = 0; i < k.size(); i++) k[i].fill((uint8_t)(0x21 + i));
  std::vector<Message> a, b;
  for (int i = 0; i < 3; i++) {
    a.emplace_back(Bytes(300 * i + 1, (uint8_t)(0x40 + i)));
    b.emplace_back(a.back().msg);
  }
  const std::vector<Message> plain = a;
  EXPECT(!eng.key_encrypt(a, key, 512, &k));
  EXPECT(!eng.key_encrypt(b, std::vector<AffinePoint>(b.size(), pub), 512, &k));
  for (size_t i = 0; i < a.size(); i++)
    EXPECT(a[i].msg == b[i].msg && a[i].digest == b[i].digest && a[i].asym_nonce == b[i].asym_nonce);
  auto dec = eng.key_decrypt(a, std::vector<Bytes>(a.size(), pws[0]));
  for (size_t i = 0; i < a.size(); i++) EXPECT(!dec[i] && a[i].msg == plain[i].msg);
  // an off-curve point is refused
  AffinePoint off = pub;
  off[60] ^= 0x10;
  bool threw = false;
  try {
    eng.prepare(off);
  } catch (const GpuError& e) {
    threw = e.status == CAPY_ERR_BAD_POINT;
  }
  EXPECT(threw);
  printf("prepared mirror ok\n");
  return 0;
}
