// tests/host/hasher_mirror_check.cpp -- the resumable streams of the C++ host mirror
// (capycrypt_b200/host/capycrypt_gpu.hpp): pieces fed through Engine::sha3_hasher / Engine::kmac_xof_hasher give what
// compute_sha3_hash / kmac_xof give for the whole messages.  Needs a GPU; compiled and run by tests/test_hasher_gpu.py.
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
  std::vector<Bytes> keys = {Bytes(131, 0x42), Bytes(), Bytes(32, 0x07)};
  for (int d : {224, 256, 384, 512}) {
    std::vector<Message> ref = whole;
    EXPECT(!eng.compute_sha3_hash(ref, d));
    gpu::Hasher h = eng.sha3_hasher(n, d);
    for (size_t k = 0; k < updates; k++) h.update(pieces[k]);
    auto got = h.final();
    for (size_t i = 0; i < n; i++) EXPECT(got[i] == ref[i].digest);
    if (d == 224) continue;
    auto want = eng.kmac_xof(keys, whole, 1000, "My Tagged Application", d);
    gpu::Hasher km = eng.kmac_xof_hasher(keys, "My Tagged Application", d);
    for (size_t k = 0; k < updates; k++) km.update(pieces[k]);
    EXPECT(km.final(1000) == want);
    bool refused = false;
    try {
      km.update(pieces[0]);
    } catch (const GpuError& e) {
      refused = e.status == CAPY_ERR_BAD_ARG;
    }
    EXPECT(refused);
  }
  bool refused = false;
  try {
    eng.kmac_xof_hasher(keys, "", 224);
  } catch (const GpuError& e) {
    refused = e.status == CAPY_ERR_BAD_ARG;
  }
  EXPECT(refused);
  printf("OK\n");
  return 0;
}
