// tests/host/ed448_prepared_host_check.cpp -- TEST SCAFFOLDING for prepared public keys.  Compiles the engine's
// __host__ __device__ comb code (capycrypt_b200/csrc/ed448.cuh) for the CPU: the window builder for any point, the
// conversion of affine multiples into table entries that fb_table_kernel runs, and the single and joint combs.
// Built and loaded by tests/test_ed448_prepared_host.py; never part of libcapycrypt_gpu.so.
#include <cstdint>
#include <cstring>

#include "../../capycrypt_b200/csrc/ed448.cuh"

using namespace capy;

static void pt_in(PtExt& p, const uint8_t* xy) {
  uint32_t w[14];
  Fe x, y;
  memcpy(w, xy, 56);
  fe_from_words(x, w);
  memcpy(w, xy + 56, 56);
  fe_from_words(y, w);
  pt_from_affine(p, x, y);
}
static void pt_out(uint8_t* xy, const PtExt& p) {
  Fe zi, x, y;
  fe_inv(zi, p.Z);
  fe_mul(x, p.X, zi);
  fe_mul(y, p.Y, zi);
  uint32_t w[14];
  fe_to_words(w, x);
  memcpy(xy, w, 56);
  fe_to_words(w, y);
  memcpy(xy + 56, w, 56);
}
static constexpr size_t kRow = (size_t)FB_ENTRIES * FB_ENTRY_WORDS;

extern "C" {
size_t host_table_words() { return (size_t)FB_WINDOWS * kRow; }

// G's table as the library builds it (fb_table_kernel without points)
void host_table_g(uint32_t* table) {
  for (int i = 0; i < FB_WINDOWS; i++) fb_build_window(table + i * kRow, i);
}
// the window builder given the point P (affine bytes)
void host_table_of(const uint8_t* xy, uint32_t* table) {
  PtExt p;
  pt_in(p, xy);
  for (int i = 0; i < FB_WINDOWS; i++) fb_build_window(table + i * kRow, i, p);
}
// fb_table_kernel with points: entry t from the affine point t (t = 16 i + j)
void host_table_from_points(const uint8_t* points_xy, uint32_t* table) {
  for (int t = 0; t < FB_WINDOWS * FB_ENTRIES; t++) fb_niels_entry_xy(table + (size_t)t * FB_ENTRY_WORDS, points_xy + 112 * t);
}
// [k mod r]P over P's table
void host_comb(const uint8_t* k_be, const uint32_t* table, int constant_time, uint8_t* out_xy) {
  Sc k, kr;
  sc_from_be(k, k_be);
  sc_reduce_448(kr, k);
  PtExt r;
  pt_fixed_base_mul(r, kr, table, constant_time != 0);
  pt_out(out_xy, r);
}
// [z mod r]G + [h mod r]V: the joint comb of a prepared verification
void host_joint_comb(const uint8_t* z_be, const uint8_t* h_be, const uint32_t* table_g, const uint32_t* table_v,
                     int constant_time, uint8_t* out_xy) {
  Sc z, zr, h, hr;
  sc_from_be(z, z_be);
  sc_reduce_448(zr, z);
  sc_from_be(h, h_be);
  sc_reduce_448(hr, h);
  PtExt r;
  pt_fixed_base_mul(r, zr, table_g, constant_time != 0, &hr, table_v);
  pt_out(out_xy, r);
}
}
