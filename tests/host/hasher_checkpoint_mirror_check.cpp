// tests/host/hasher_checkpoint_mirror_check.cpp -- checkpoints and forks of the C++ host mirror
// (capycrypt_b200/host/capycrypt_gpu.hpp): a stream exported by Hasher::export_blob and resumed by Engine::import_hasher
// in another Engine, or forked by Hasher::fork, gives what compute_sha3_hash / kmac_xof give for the whole messages.
// Needs a GPU; compiled and run by tests/test_hasher_checkpoint_gpu.py.
#include <cstdio>
#include "../../capycrypt_b200/host/capycrypt_gpu.hpp"
using namespace capycrypt;

#define EXPECT(c) do { if (!(c)) { printf("FAIL line %d: %s\n", __LINE__, #c); return 1; } } while (0)

int main() {
  const size_t n = 3;
  // item i: a head of (53 i + 70) bytes before the checkpoint and a tail of (41 i + 90) bytes after it
  std::vector<Bytes> head(n), tail(n);
  std::vector<Message> whole(n);
  for (size_t i = 0; i < n; i++) {
    for (size_t b = 0; b < 53 * i + 70; b++) head[i].push_back((uint8_t)(i * 17 + b));
    for (size_t b = 0; b < 41 * i + 90; b++) tail[i].push_back((uint8_t)(i * 29 + 3 * b));
    whole[i].msg = head[i];
    whole[i].msg.insert(whole[i].msg.end(), tail[i].begin(), tail[i].end());
  }
  std::vector<Message> heads(n);
  for (size_t i = 0; i < n; i++) heads[i].msg = head[i];
  const std::vector<Bytes> keys = {Bytes(131, 0x42), Bytes(), Bytes(32, 0x07)};
  gpu::Engine a, b;
  for (int d : {224, 256, 512}) {
    std::vector<Message> ref = whole, ref_head = heads;
    EXPECT(!a.compute_sha3_hash(ref, d));
    EXPECT(!a.compute_sha3_hash(ref_head, d));
    Bytes blob;
    {
      gpu::Hasher h = a.sha3_hasher(n, d);
      h.update(head);
      blob = h.export_blob();
      gpu::Hasher so_far = h.fork({0, 1, 2});  // the digest so far; h goes on
      auto mid = so_far.final();
      for (size_t i = 0; i < n; i++) EXPECT(mid[i] == ref_head[i].digest);
      gpu::Hasher rev = h.fork({2, 1, 0, 0});
      rev.update({tail[2], tail[1], tail[0], tail[0]});
      auto r = rev.final();
      EXPECT(r[0] == ref[2].digest && r[1] == ref[1].digest && r[2] == ref[0].digest && r[3] == ref[0].digest);
      h.update(tail);
      auto got = h.final();
      for (size_t i = 0; i < n; i++) EXPECT(got[i] == ref[i].digest);
      bool refused = false;  // a finished hasher cannot be exported
      try {
        h.export_blob();
      } catch (const GpuError& e) {
        refused = e.status == CAPY_ERR_BAD_ARG;
      }
      EXPECT(refused);
    }
    gpu::Hasher r = b.import_hasher(blob);  // another Engine
    r.update(tail);
    auto got = r.final();
    for (size_t i = 0; i < n; i++) EXPECT(got[i] == ref[i].digest);
    if (d == 224) continue;
    auto want = a.kmac_xof(keys, whole, 1000, "My Tagged Application", d);
    gpu::Hasher km = a.kmac_xof_hasher(keys, "My Tagged Application", d);
    km.update(head);
    gpu::Hasher kr = b.import_hasher(km.export_blob());
    kr.update(tail);
    EXPECT(kr.final(1000) == want);
  }
  bool refused = false;
  try {
    Bytes junk(64, 0);
    b.import_hasher(junk);
  } catch (const GpuError& e) {
    refused = e.status == CAPY_ERR_BAD_ARG;
  }
  EXPECT(refused);
  printf("OK\n");
  return 0;
}
