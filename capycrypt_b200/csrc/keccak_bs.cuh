// keccak_bs.cuh -- Keccak-f[1600] bitsliced across the 32 messages of a warp.
//
// Bit m of every register belongs to message m of the warp, so each register holds one bit position of one lane
// for 32 messages.  Thread t holds bit positions z = 2t (word 0) and z = 2t + 1 (word 1) of all 25 lanes: 50 words.
// A rotation by r then moves whole words between threads and needs no bit arithmetic (bit z of the result is bit
// z - r of the input):
//   r even: both words come from thread t - r/2, same word;
//   r odd:  word 0 takes word 1 of thread t - (r+1)/2, word 1 takes word 0 of thread t - (r-1)/2.
// Pi is register renaming, theta and chi stay one 3-input LOP3 per word.  Per round: 20 + 50 + 50 LOP3 plus iota
// on the ALU pipe, 5 (theta) + 47 (rho) shuffles on the shuffle unit, which the one-state-per-thread form
// (keccak.cuh) leaves idle while it spends 58 funnel shifts per round on the ALU pipe.
//
// Every function here shuffles with a full mask: all 32 threads of the warp must call it together.
#pragma once
#include <cstdint>

#include "keccak.cuh"

namespace capy {

// bit z of RC[r] for z = 2t (x) and z = 2t + 1 (y), as a mask over the rounds r: bit r = bit z of RC[r]
static __device__ const uint2 KECCAK_RC_BITS[32] = {
    {0x50F4F1u, 0x0DB916u}, {0x000000u, 0x8C7F94u}, {0x000000u, 0x000000u}, {0x000000u, 0x327356u},
    {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0xB5D4DEu},
    {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u},
    {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0xD81C68u},
    {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u},
    {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u},
    {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u},
    {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0x000000u}, {0x000000u, 0xBBE0CCu}};

// v of thread lane - K (mod 32): shfl reads bits 4:0 of the source lane, so the subtraction may wrap
template <int K>
__device__ __forceinline__ uint32_t bs_from(uint32_t v, uint32_t lane) {
  if constexpr (K % 32 == 0) return v;
  else return __shfl_sync(0xffffffffu, v, (int)(lane - (uint32_t)K));
}

// b := rotl64(t, R) in the bitsliced layout
template <int R>
__device__ __forceinline__ void bs_rot(uint32_t (&b)[2], uint32_t t0, uint32_t t1, uint32_t lane) {
  if constexpr (R % 2 == 0) {
    b[0] = bs_from<R / 2>(t0, lane);
    b[1] = bs_from<R / 2>(t1, lane);
  } else {
    b[0] = bs_from<(R + 1) / 2>(t1, lane);
    b[1] = bs_from<(R - 1) / 2>(t0, lane);
  }
}

// as CAPY_RHO_PI in keccak.cuh: B[y][2x+3y] = rot(A[x][y] ^ C[x-1] ^ rot1(C[x+1]), rho[x][y]); n[x] = rot1(C[x])
#define CAPY_BS_RHO_PI(X, Y, R)                                                                       \
  bs_rot<(R)>(b[(Y) + 5 * ((2 * (X) + 3 * (Y)) % 5)],                                                 \
              lop_xor3(a[(X) + 5 * (Y)][0], c[((X) + 4) % 5][0], n[((X) + 1) % 5][0]),                \
              lop_xor3(a[(X) + 5 * (Y)][1], c[((X) + 4) % 5][1], n[((X) + 1) % 5][1]), lane);

// ~v where (rounds & round) != 0: a predicate test and a predicated NOT, two ALU instructions
__device__ __forceinline__ uint32_t bs_flip_if(uint32_t v, uint32_t rounds, uint32_t round) {
  asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\t@p not.b32 %0, %0;\n\t}"
      : "+r"(v)
      : "r"(rounds), "r"(round));
  return v;
}

// one round; rc: bits 2t / 2t+1 of the round constants (KECCAK_RC_BITS[t]), round: 1 << r
__device__ __forceinline__ void keccak_bs_round(uint32_t (&a)[25][2], uint32_t lane, uint2 rc, uint32_t round) {
  uint32_t c[5][2], n[5][2], b[25][2];
#pragma unroll
  for (int x = 0; x < 5; x++) {
#pragma unroll
    for (int h = 0; h < 2; h++) c[x][h] = lop_xor3(lop_xor3(a[x][h], a[x + 5][h], a[x + 10][h]), a[x + 15][h], a[x + 20][h]);
    n[x][0] = bs_from<1>(c[x][1], lane);  // bit 2t - 1 lives in word 1 of thread t - 1
    n[x][1] = c[x][0];
  }
  CAPY_BS_RHO_PI(0, 0, 0)  CAPY_BS_RHO_PI(1, 0, 1)  CAPY_BS_RHO_PI(2, 0, 62) CAPY_BS_RHO_PI(3, 0, 28) CAPY_BS_RHO_PI(4, 0, 27)
  CAPY_BS_RHO_PI(0, 1, 36) CAPY_BS_RHO_PI(1, 1, 44) CAPY_BS_RHO_PI(2, 1, 6)  CAPY_BS_RHO_PI(3, 1, 55) CAPY_BS_RHO_PI(4, 1, 20)
  CAPY_BS_RHO_PI(0, 2, 3)  CAPY_BS_RHO_PI(1, 2, 10) CAPY_BS_RHO_PI(2, 2, 43) CAPY_BS_RHO_PI(3, 2, 25) CAPY_BS_RHO_PI(4, 2, 39)
  CAPY_BS_RHO_PI(0, 3, 41) CAPY_BS_RHO_PI(1, 3, 45) CAPY_BS_RHO_PI(2, 3, 15) CAPY_BS_RHO_PI(3, 3, 21) CAPY_BS_RHO_PI(4, 3, 8)
  CAPY_BS_RHO_PI(0, 4, 18) CAPY_BS_RHO_PI(1, 4, 2)  CAPY_BS_RHO_PI(2, 4, 61) CAPY_BS_RHO_PI(3, 4, 56) CAPY_BS_RHO_PI(4, 4, 14)
#pragma unroll
  for (int y = 0; y < 5; y++) {
#pragma unroll
    for (int x = 0; x < 5; x++) {
#pragma unroll
      for (int h = 0; h < 2; h++)
        a[x + 5 * y][h] = lop_chi(b[x + 5 * y][h], b[(x + 1) % 5 + 5 * y][h], b[(x + 2) % 5 + 5 * y][h]);
    }
  }
  a[0][0] = bs_flip_if(a[0][0], rc.x, round);
  a[0][1] = bs_flip_if(a[0][1], rc.y, round);
}
#undef CAPY_BS_RHO_PI

// 32 x 32 bit transpose across the warp: bit j of thread i becomes bit i of thread j.  Five butterfly stages; stage d
// swaps thread-index bit d with bit-position bit d.  BsTranspose holds the per-thread rotation and keep-mask of each
// stage, so a stage is one shuffle, one funnel shift and one LOP3.
struct BsTranspose {
  uint32_t rot[5], keep[5];
  __device__ __forceinline__ explicit BsTranspose(uint32_t lane) {
#pragma unroll
    for (int k = 0; k < 5; k++) {
      const uint32_t d = 16u >> k;
      const uint32_t lo_bits = k == 0 ? 0x0000FFFFu : k == 1 ? 0x00FF00FFu : k == 2 ? 0x0F0F0F0Fu : k == 3 ? 0x33333333u : 0x55555555u;
      const bool upper = lane & d;
      // the lower thread takes the partner's bits B - d into its bits B with bit d set, the upper one the partner's
      // bits B + d into its bits B with bit d clear
      rot[k] = upper ? 32u - d : d;
      keep[k] = upper ? ~lo_bits : lo_bits;
    }
  }
  __device__ __forceinline__ uint32_t operator()(uint32_t x) const {
#pragma unroll
    for (int k = 0; k < 5; k++) {
      const uint32_t y = __shfl_xor_sync(0xffffffffu, x, 16u >> k);
      const uint32_t r = __funnelshift_l(y, y, rot[k]);
      // (x & keep) | (r & ~keep) as one LOP3; written out, it is compiled as three
      asm("lop3.b32 %0, %0, %1, %2, 0xE4;" : "+r"(x) : "r"(r), "r"(keep[k]));
    }
    return x;
  }
};

// Thread j holds bit z = j of a lane in lo and z = 32 + j in hi (a transposed 64-bit word); w receives bits 2t, 2t+1.
__device__ __forceinline__ void bs_gather(uint32_t (&w)[2], uint32_t lo, uint32_t hi, uint32_t lane) {
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int src = (int)(2 * lane + h);  // bits 4:0: thread 2t + h of the low or the high half
    const uint32_t l = __shfl_sync(0xffffffffu, lo, src);
    const uint32_t u = __shfl_sync(0xffffffffu, hi, src);
    w[h] = lane < 16 ? l : u;
  }
}

// the inverse of bs_gather: lo / hi receive bits z = j / 32 + j of the lane in thread j
__device__ __forceinline__ void bs_scatter(uint32_t& lo, uint32_t& hi, const uint32_t (&w)[2], uint32_t lane) {
  const int src = (int)(lane >> 1);
  const uint32_t l0 = __shfl_sync(0xffffffffu, w[0], src), l1 = __shfl_sync(0xffffffffu, w[1], src);
  const uint32_t u0 = __shfl_sync(0xffffffffu, w[0], src + 16), u1 = __shfl_sync(0xffffffffu, w[1], src + 16);
  lo = lane & 1 ? l1 : l0;
  hi = lane & 1 ? u1 : u0;
}

}  // namespace capy
