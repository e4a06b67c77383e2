// ed448.cuh -- Ed448-Goldilocks group arithmetic for sm_100a (untwisted Edwards curve
// x^2 + y^2 = 1 + d x^2 y^2, d = -39081, a = 1; SURVEY.md App. C.2).
//
// Replaces `ExtendedPoint::{generator, Mul<Scalar>, Add, to_affine}` of the un-vendored crate
// tiny_ed448_goldilocks 0.1.8 (call sites ecc/keypair.rs:44, ecc/signable.rs:48-49,77,
// ecc/encryptable.rs:37-38,78).  Extended coordinates (X:Y:Z:T), complete formulas
// (add-2008-hwcd / dbl-2008-hwcd with a = 1; d is a non-square so the unified addition has no
// exceptional points), so every input -- identity, small-order points, P + P -- takes the same path.
//
// Scalar multiplication is a fixed-window ladder on signed radix-16 digits:
//   fixed base   on the 4-isogenous twisted curve: 90 windows x 16 Niels entries (j+1) * 32^i * phi(G)
//                -> 90 mixed additions of 7 M, no doubling, dual isogeny back to E at the end
//   variable     per-item table 1P..8P, 113 windows x (4 doublings + 1 addition)
// Table entries are chosen by a constant-time scan (every entry is read, the wanted one is kept
// with a mask) unless the caller states that the scalar is public (verify).
#pragma once
#include "fp448.cuh"
#include "sc448.cuh"

namespace capy {

constexpr uint32_t EDW_D_ABS = 39081u;  // d = -39081

struct PtExt {  // extended projective, all coordinates tight
  Fe X, Y, Z, T;
};
struct PtCached {  // projective table entry: X, Y, Z, Td = d*T
  Fe X, Y, Z, Td;
};

CAPY_HD void pt_identity(PtExt& p) {
  fe_zero(p.X);
  fe_one(p.Y);
  fe_one(p.Z);
  fe_zero(p.T);
}

// r = d * a = -(39081 * a)
CAPY_HD void fe_mul_d(Fe& r, const Fe& a) {
  uint64_t R[16];
#pragma unroll
  for (int i = 0; i < 16; i++) R[i] = (uint64_t)a.v[i] * EDW_D_ABS;
  Fe t;
  fe_carry_wide(t, R);
  fe_neg(r, t);
}

// shared tail of the additions: given A = X1*X2, B = Y1*Y2, C = d*T1*T2, D = Z1*Z2 (tight) and
// E0 = (X1+Y1)*(X2+Y2) (tight):  E = E0 - A - B, F = D - C, G = D + C, H = B - A  (a = 1)
template <bool WANT_T>
CAPY_HD void add_tail(PtExt& r, const Fe& A, const Fe& B, const Fe& C, const Fe& D, const Fe& E0) {
  Fe E, F, G, H, AB;
  fe_add(AB, A, B);     // alpha 2
  fe_sub4(E, E0, AB);   // alpha 5
  fe_weak(E);           // tight
  fe_sub(F, D, C);      // alpha 3
  fe_add(G, D, C);      // alpha 2
  fe_sub(H, B, A);      // alpha 3
  fe_mul(r.X, E, F);    // 1 x 3
  fe_mul(r.Y, G, H);    // 2 x 3
  fe_mul(r.Z, F, G);    // 3 x 2
  if (WANT_T) fe_mul(r.T, E, H);  // 1 x 3
}

// r = p + q, q a projective table entry: 9 M
template <bool WANT_T>
CAPY_HD void pt_add_cached(PtExt& r, const PtExt& p, const PtCached& q) {
  Fe A, B, C, D, E0, s1, s2;
  fe_mul(A, p.X, q.X);
  fe_mul(B, p.Y, q.Y);
  fe_mul(C, p.T, q.Td);
  fe_mul(D, p.Z, q.Z);
  fe_add(s1, p.X, p.Y);
  fe_add(s2, q.X, q.Y);
  fe_mul(E0, s1, s2);
  add_tail<WANT_T>(r, A, B, C, D, E0);
}

// r = 2p: 4 S + 3 M (+1 M for T).  Does not read p.T.
template <bool WANT_T>
CAPY_HD void pt_double(PtExt& r, const PtExt& p) {
  Fe A, B, C, E, F, G, H, s, ZZ;
  fe_sqr(A, p.X);
  fe_sqr(B, p.Y);
  fe_sqr(ZZ, p.Z);
  fe_add(s, p.X, p.Y);   // alpha 2
  fe_sqr(E, s);          // 2 x 2
  fe_add(G, A, B);       // alpha 2
  fe_sub4(E, E, G);      // alpha 5
  fe_weak(E);            // tight
  fe_add(C, ZZ, ZZ);     // alpha 2
  fe_sub4(F, G, C);      // alpha 6
  fe_weak(F);            // tight
  fe_sub(H, A, B);       // alpha 3
  fe_mul(r.X, E, F);     // 1 x 1
  fe_mul(r.Y, G, H);     // 2 x 3
  fe_mul(r.Z, F, G);     // 1 x 2
  if (WANT_T) fe_mul(r.T, E, H);  // 1 x 3
}

CAPY_HD void pt_to_cached(PtCached& c, const PtExt& p) {
  fe_copy(c.X, p.X);
  fe_copy(c.Y, p.Y);
  fe_copy(c.Z, p.Z);
  fe_mul_d(c.Td, p.T);
}

// affine (x, y) -> extended; returns false when the point is not on the curve
CAPY_HD bool pt_from_affine(PtExt& p, const Fe& x, const Fe& y) {
  fe_copy(p.X, x);
  fe_copy(p.Y, y);
  fe_one(p.Z);
  fe_mul(p.T, x, y);
  // x^2 + y^2 - 1 + 39081 x^2 y^2 == 0
  Fe x2, y2, l, m, one;
  fe_sqr(x2, x);
  fe_sqr(y2, y);
  fe_mul(m, x2, y2);
  fe_mul_d(m, m);        // d x^2 y^2 (tight)
  fe_add(l, x2, y2);     // alpha 2
  fe_one(one);
  fe_add(m, m, one);     // 1 + d x^2 y^2, alpha ~1
  fe_sub(l, l, m);       // alpha 4
  return fe_is_zero(l);
}

// ---- fixed-base comb on the 4-isogenous twisted curve ------------------------------------------------
// [k]G is computed as  phi^([k / 4 mod r] * phi(G))  where phi: E -> E' is the 4-isogeny onto the twisted
// Edwards curve E': -x^2 + y^2 = 1 + (d - 1) x^2 y^2 and phi^ its dual (phi^ o phi = [4]; G has odd order r,
// so this is exact).  On E' (a = -1) a mixed addition with a precomputed Niels entry (y - x, y + x, 2 d' x y)
// costs 7 M instead of 8 M on E.  Signed radix-32 digits: 90 windows x 16 entries = 270 KB table, 90 mixed
// additions and no doubling per scalar multiplication.
#ifndef CAPY_FB_WBITS
#define CAPY_FB_WBITS 5  // measured: 4 / 5 / 6 bits -> see profiles/README.md round 2 (scan cost against additions)
#endif
constexpr int FB_WBITS = CAPY_FB_WBITS;
constexpr int FB_WINDOWS = (447 + FB_WBITS - 1) / FB_WBITS;  // kq < r < 2^446, one more bit for the signed recoding
constexpr int FB_ENTRIES = 1 << (FB_WBITS - 1);
constexpr int FB_ENTRY_WORDS = 48;  // ymx | ypx | td2, 16 canonical limbs each
constexpr uint32_t EDW_2D_TW_ABS = 2u * 39082u;  // 2 d' = -78164

struct PtNiels {  // affine point of E' as (y - x, y + x, 2 d' x y)
  Fe ymx, ypx, td2;
};

#if defined(__CUDA_ARCH__)
#define CAPY_LD128(p) __ldg(reinterpret_cast<const uint4*>(p))
#else
#define CAPY_LD128(p) (*reinterpret_cast<const uint4*>(p))
#endif

// r = p + q on E' (a = -1), q affine Niels: 7 M (add-2008-hwcd-3 with Z2 = 1)
template <bool WANT_T>
CAPY_HD void pt_madd_tw(PtExt& r, const PtExt& p, const PtNiels& q) {
  Fe A, B, C, D, E, F, G, H, t0, t1;
  fe_sub(t0, p.Y, p.X);      // alpha 3
  fe_add(t1, p.Y, p.X);      // alpha 2
  fe_mul(A, t0, q.ymx);      // 3 x 1
  fe_mul(B, t1, q.ypx);      // 2 x 1
  fe_mul(C, p.T, q.td2);     // 1 x 2 (td2 may be an unreduced negation)
  fe_add(D, p.Z, p.Z);       // alpha 2
  fe_sub(E, B, A);           // alpha 3
  fe_add(H, B, A);           // alpha 2
  fe_sub(F, D, C);           // alpha 4
  fe_weak(F);                // tight
  fe_add(G, D, C);           // alpha 3
  fe_mul(r.X, E, F);         // 3 x 1
  fe_mul(r.Y, G, H);         // 3 x 2
  fe_mul(r.Z, F, G);         // 1 x 3
  if (WANT_T) fe_mul(r.T, E, H);  // 3 x 2
}

// e = |dgt| * 32^i * phi(G) with the sign applied; dgt == 0 gives the identity (1, 1, 0).
// `row` = the 16 entries of window i.  STAGED: the row sits in shared memory (plain loads, broadcast);
// otherwise it is read from global memory through the read-only path.
template <bool STAGED>
CAPY_HD void fb_lookup_row(PtNiels& e, const uint32_t* __restrict__ row, int dgt, bool CONSTANT_TIME) {
  const uint32_t neg = dgt < 0 ? 0xffffffffu : 0u;
  const uint32_t mag = (uint32_t)(dgt < 0 ? -dgt : dgt);  // 0..16
  uint32_t w[FB_ENTRY_WORDS];
#pragma unroll
  for (int k = 0; k < FB_ENTRY_WORDS; k++) w[k] = 0;
  w[0] = 1;   // y - x = 1
  w[16] = 1;  // y + x = 1
  if (CONSTANT_TIME) {
#pragma unroll 1
    for (uint32_t j = 1; j <= FB_ENTRIES; j++) {
      const uint32_t m = (j == mag) ? 0xffffffffu : 0u;
      const uint32_t* ent = row + (j - 1) * FB_ENTRY_WORDS;
#pragma unroll
      for (int k = 0; k < FB_ENTRY_WORDS; k += 4) {
        const uint4 v = STAGED ? *reinterpret_cast<const uint4*>(ent + k) : CAPY_LD128(ent + k);
        w[k + 0] = (v.x & m) | (w[k + 0] & ~m);
        w[k + 1] = (v.y & m) | (w[k + 1] & ~m);
        w[k + 2] = (v.z & m) | (w[k + 2] & ~m);
        w[k + 3] = (v.w & m) | (w[k + 3] & ~m);
      }
    }
  } else if (mag != 0) {
    const uint32_t* ent = row + (mag - 1) * FB_ENTRY_WORDS;
#pragma unroll
    for (int k = 0; k < FB_ENTRY_WORDS; k += 4) {
      const uint4 v = STAGED ? *reinterpret_cast<const uint4*>(ent + k) : CAPY_LD128(ent + k);
      w[k + 0] = v.x;
      w[k + 1] = v.y;
      w[k + 2] = v.z;
      w[k + 3] = v.w;
    }
  }
  // -(x, y) = (-x, y): swap (y - x) <-> (y + x), negate 2 d' x y (left unreduced: 2p - td2, alpha 2)
#pragma unroll
  for (int k = 0; k < 16; k++) {
    const uint32_t t = (w[k] ^ w[16 + k]) & neg;
    e.ymx.v[k] = w[k] ^ t;
    e.ypx.v[k] = w[16 + k] ^ t;
    const uint32_t ntd = (k == 8 ? 2u * (M28 - 1u) : 2u * M28) - w[32 + k];
    e.td2.v[k] = (ntd & neg) | (w[32 + k] & ~neg);
  }
}

// signed radix-32 digit i of kq (with the running carry of the recoding)
CAPY_HD int fb_digit(const Sc& kq, int i, uint32_t& carry) {
  const int bit = FB_WBITS * i, q = bit >> 5, sh = bit & 31;
  uint32_t v = kq.w[q] >> sh;
  if (sh > 32 - FB_WBITS && q + 1 < 14) v |= kq.w[q + 1] << (32 - sh);
  const uint32_t win = (v & ((1u << FB_WBITS) - 1u)) + carry;
  carry = win >= (1u << (FB_WBITS - 1)) ? 1u : 0u;
  return (int)win - (int)(carry << FB_WBITS);
}

// dual isogeny phi^: E' -> E on projective coordinates, result extended on E:
//   x = 2XY / (Y^2 + X^2),  y = (Y^2 - X^2) / (2Z^2 - Y^2 + X^2)
CAPY_HD void pt_dual_isogeny(PtExt& r, const PtExt& p) {
  Fe A, B, ZZ, XY, xn, xd, yn, yd;
  fe_sqr(A, p.X);
  fe_sqr(B, p.Y);
  fe_sqr(ZZ, p.Z);
  fe_mul(XY, p.X, p.Y);
  fe_add(xn, XY, XY);    // alpha 2
  fe_add(xd, B, A);      // alpha 2
  fe_sub(yn, B, A);      // alpha 3
  fe_add(yd, ZZ, ZZ);    // alpha 2
  fe_sub4(yd, yd, yn);   // alpha 6
  fe_weak(yd);           // tight
  fe_mul(r.X, xn, yd);   // 2 x 1
  fe_mul(r.Y, yn, xd);   // 3 x 2
  fe_mul(r.Z, xd, yd);   // 2 x 1
  fe_mul(r.T, xn, yn);   // 2 x 3
}

// r = [k]P (extended, on E) for k in [0, r) via the comb table of phi(P) read from global memory; with table2 the
// windows of k2 over table2 (the comb table of phi(Q)) run into the same accumulator: r = [k]P + [k2]Q.  Exact when
// P and Q both have odd order r.  (The CUDA kernel in ed448_fixed.cu runs the same loop with the table rows staged
// through shared memory.)
CAPY_HD void pt_fixed_base_mul(PtExt& r, const Sc& k, const uint32_t* __restrict__ table, bool CONSTANT_TIME,
                               const Sc* k2 = nullptr, const uint32_t* __restrict__ table2 = nullptr) {
  const Sc inv4 = {CAPY_INV4_LIMBS};
  PtExt acc;
  pt_identity(acc);  // (0, 1) is the identity of E' too
#pragma unroll 1
  for (int pass = 0; pass < (table2 ? 2 : 1); pass++) {
    const uint32_t* tab = pass ? table2 : table;
    Sc kq;
    sc_mul_mod(kq, pass ? *k2 : k, inv4);  // k / 4 mod r
    uint32_t carry = 0;
#pragma unroll 1
    for (int i = 0; i < FB_WINDOWS; i++) {
      const int dgt = fb_digit(kq, i, carry);
      PtNiels e;
      fb_lookup_row<false>(e, tab + (size_t)i * FB_ENTRIES * FB_ENTRY_WORDS, dgt, CONSTANT_TIME);
      pt_madd_tw<true>(acc, acc, e);
    }
  }
  pt_dual_isogeny(r, acc);
}

// ---- variable base ------------------------------------------------------------------------------
// [k]P for the exact integer k < 2^448 (NOT reduced: quirk Q10, ecc/signable.rs:76-77), signed radix-16 fixed
// window, per-item table 1P..8P.  The table lives in memory the caller provides (the CUDA kernel: shared memory,
// thread-interleaved).  An entry is a cached point (X, Y, Z, d*T) with every coordinate carried to its exact
// 448-bit value and packed into 14 words: 56 words = 14 uint4 chunks; chunk c of entry e sits at
// col[(e * 14 + c) * STRIDE], where col already points at this item's column.
//
// The whole computation is ONE loop whose body holds one copy of the doubling (4 S + 3 M, + 1 M for T in the last of a
// window) and one copy of the addition (8 M, + 1 M for T where an addition follows), all multiplications inlined: table construction (2P = dbl, jP = (j-1)P + P), the 113 windows
// (4 doublings + 1 addition of a looked-up entry) and the optional addend of verify (U = [z]G + [h]V,
// ecc/signable.rs:77) are iterations of that loop with different operands, so the accumulator never leaves the
// registers and no multiplication goes through an out-of-line call.
// The signed digits are not stored: with K = k + 0x888...8 (112 nibbles) digit i is nibble i of K minus 8 (the
// digits in [-8, 7] a carry recoding gives; the last one, digit 112, is 0 or 1); K sits in 15 registers and is shifted left by one nibble per
// window, so the current digit is always at bit 448.
constexpr int VB_ENTRIES = 8;
constexpr int VB_CHUNKS = 14;  // uint4 chunks per entry: X | Y | Z | d*T, 14 words each

#if defined(__CUDA_ARCH__)
// With the table in local memory (round 1) a block barrier in front of every doubling / addition paid off: the warps of
// a block fetched one instruction stream.  Since the table moved to shared memory / the L2 the barrier costs more than
// the drift (29.5 against 31.2 ms per 2^18 items, profiles/README.md round 2): off unless CAPY_VB_SYNC is defined.
#if defined(CAPY_VB_SYNC)
#define CAPY_BLOCK_SYNC() __syncthreads()
#else
#define CAPY_BLOCK_SYNC() ((void)0)
#endif
CAPY_HD uint32_t capy_fshr(uint32_t lo, uint32_t hi, uint32_t sh) { return __funnelshift_r(lo, hi, sh); }
CAPY_HD uint32_t capy_fshl(uint32_t lo, uint32_t hi, uint32_t sh) { return __funnelshift_l(lo, hi, sh); }
#else
#define CAPY_BLOCK_SYNC() ((void)0)
CAPY_HD uint32_t capy_fshr(uint32_t lo, uint32_t hi, uint32_t sh) { return (uint32_t)((((uint64_t)hi << 32) | lo) >> sh); }
CAPY_HD uint32_t capy_fshl(uint32_t lo, uint32_t hi, uint32_t sh) { return (uint32_t)(((((uint64_t)hi << 32) | lo) << sh) >> 32); }
#endif

// tight limbs -> the exact 448-bit value in limbs < 2^28 (not necessarily < p): two serial passes; the second
// cannot carry out (value < 2^448 (1 + 2^-18): after a wrap the value is tiny)
CAPY_HD void fe_carry_exact(Fe& a) {
#pragma unroll
  for (int pass = 0; pass < 2; pass++) {
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
      const uint32_t v = a.v[i] + c;
      a.v[i] = v & M28;
      c = v >> 28;
    }
    a.v[0] += c;  // 2^448 = 2^224 + 1
    a.v[8] += c;
  }
}

// limbs < 2^28 -> 14 little-endian words at w[0..13], and back
CAPY_HD void fe_pack14(uint32_t* w, const Fe& a) {
#pragma unroll
  for (int q = 0; q < 14; q++) w[q] = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) {
    const int bit = 28 * i, q = bit >> 5, sh = bit & 31;
    w[q] |= a.v[i] << sh;
    if (sh > 4 && q + 1 < 14) w[q + 1] |= a.v[i] >> (32 - sh);
  }
}
CAPY_HD void fe_unpack14(Fe& r, const uint32_t* w) {
#pragma unroll
  for (int i = 0; i < 16; i++) {
    const int bit = 28 * i, q = bit >> 5, sh = bit & 31;
    uint32_t v;
    if (sh == 0) v = w[q];
    else if (sh > 4 && q + 1 < 14) v = capy_fshr(w[q], w[q + 1], sh);
    else v = w[q] >> sh;
    r.v[i] = v & M28;
  }
}

// entry e of this item := cached form of p (X, Y, Z, d*T)
template <int STRIDE>
CAPY_HD void vb_store_entry(uint4* col, int e, const PtExt& p) {
  uint32_t w[56];
  Fe t;
  fe_copy(t, p.X);
  fe_carry_exact(t);
  fe_pack14(w, t);
  fe_copy(t, p.Y);
  fe_carry_exact(t);
  fe_pack14(w + 14, t);
  fe_copy(t, p.Z);
  fe_carry_exact(t);
  fe_pack14(w + 28, t);
  fe_mul_d(t, p.T);
  fe_carry_exact(t);
  fe_pack14(w + 42, t);
  uint4* ent = col + (size_t)e * VB_CHUNKS * STRIDE;
#pragma unroll
  for (int c = 0; c < VB_CHUNKS; c++) {
    uint4 v;
    v.x = w[4 * c];
    v.y = w[4 * c + 1];
    v.z = w[4 * c + 2];
    v.w = w[4 * c + 3];
    ent[c * STRIDE] = v;
  }
}

// e = dgt * P from the table (dgt in [-8, 8]); constant time = every entry is read and the wanted one kept with a
// mask.  The negation -(X : Y : Z : T) = (-X : Y : Z : -T) is left unreduced (2p - v, alpha 2): the addition
// multiplies it with tight operands only.
template <int STRIDE>
CAPY_HD void vb_lookup(PtCached& e, const uint4* col, int dgt, bool CONSTANT_TIME) {
  const uint32_t neg = dgt < 0 ? 0xffffffffu : 0u;
  const uint32_t mag = (uint32_t)(dgt < 0 ? -dgt : dgt);
  uint32_t w[56];
  if (CONSTANT_TIME) {
#pragma unroll
    for (int k = 0; k < 56; k++) w[k] = 0;
    // software pipeline over half entries (7 chunks): the loads of the next half are in flight while the current one is
    // masked in -- the second four warps of a block read their table from the L2 (~400 clocks per dependent batch)
    constexpr int HALF = VB_CHUNKS / 2;
    uint4 buf[2][HALF];
#pragma unroll
    for (int c = 0; c < HALF; c++) buf[0][c] = col[c * STRIDE];
#pragma unroll
    for (int hq = 0; hq < 2 * VB_ENTRIES; hq++) {
      if (hq + 1 < 2 * VB_ENTRIES) {
#pragma unroll
        for (int c = 0; c < HALF; c++) buf[(hq + 1) & 1][c] = col[(size_t)((hq + 1) * HALF + c) * STRIDE];
      }
      const uint32_t m = ((uint32_t)(hq / 2 + 1) == mag) ? 0xffffffffu : 0u;
      const int c0 = (hq & 1) * HALF;
#pragma unroll
      for (int c = 0; c < HALF; c++) {
        const uint4 v = buf[hq & 1][c];
        w[4 * (c0 + c) + 0] |= v.x & m;
        w[4 * (c0 + c) + 1] |= v.y & m;
        w[4 * (c0 + c) + 2] |= v.z & m;
        w[4 * (c0 + c) + 3] |= v.w & m;
      }
    }
  } else {
    const uint4* ent = col + (size_t)(mag ? mag - 1 : 0) * VB_CHUNKS * STRIDE;
    const uint32_t m = mag ? 0xffffffffu : 0u;
#pragma unroll
    for (int c = 0; c < VB_CHUNKS; c++) {
      const uint4 v = ent[c * STRIDE];
      w[4 * c + 0] = v.x & m;
      w[4 * c + 1] = v.y & m;
      w[4 * c + 2] = v.z & m;
      w[4 * c + 3] = v.w & m;
    }
  }
  const uint32_t one = mag ? 0u : 1u;  // digit 0: the identity (0 : 1 : 1 : 0)
  w[14] |= one;
  w[28] |= one;
  Fe x, td;
  fe_unpack14(x, w);
  fe_unpack14(e.Y, w + 14);
  fe_unpack14(e.Z, w + 28);
  fe_unpack14(td, w + 42);
#pragma unroll
  for (int i = 0; i < 16; i++) {
    const uint32_t twop = i == 8 ? 2u * (M28 - 1u) : 2u * M28;
    e.X.v[i] = ((twop - x.v[i]) & neg) | (x.v[i] & ~neg);
    e.Td.v[i] = ((twop - td.v[i]) & neg) | (td.v[i] & ~neg);
  }
}

// r = 2r (dbl-2008-hwcd, a = 1): 4 S + 3 M (+ 1 M for T), multiplications inlined
CAPY_HD void vb_double(PtExt& r, bool want_t) {
  Fe A, B, C, E, F, G, H, s, ZZ;
  fe_sqr_inl(A, r.X);
  fe_sqr_inl(B, r.Y);
  fe_sqr_inl(ZZ, r.Z);
  fe_add(s, r.X, r.Y);   // alpha 2
  fe_sqr_inl(E, s);      // 2 x 2
  fe_add(G, A, B);       // alpha 2
  fe_sub4(E, E, G);      // alpha 5
  fe_weak(E);            // tight
  fe_add(C, ZZ, ZZ);     // alpha 2
  fe_sub4(F, G, C);      // alpha 6
  fe_weak(F);            // tight
  fe_sub(H, A, B);       // alpha 3
  fe_mul_inl(r.X, E, F);
  fe_mul_inl(r.Y, G, H);
  fe_mul_inl(r.Z, F, G);
  if (want_t) fe_mul_inl(r.T, E, H);
}

// r = r + q (add-2008-hwcd, a = 1, q cached with alpha(q.X), alpha(q.Td) <= 2): 8 M (+ 1 M for T).  Ordered so that few
// field elements are live at a time (the operands of r and q die early): the inlined body fits the registers.  The
// additions of the window loop are followed by doublings, which do not read T: they skip that product.
CAPY_HD void vb_add(PtExt& r, const PtCached& q, bool want_t) {
  Fe A, B, E, H, s1, s2;
  fe_add(s1, r.X, r.Y);       // alpha 2
  fe_add(s2, q.X, q.Y);       // alpha 3
  fe_mul_inl(E, s1, s2);      // 2 x 3: (X1 + Y1)(X2 + Y2)
  fe_mul_inl(A, r.X, q.X);    // 1 x 2
  fe_mul_inl(B, r.Y, q.Y);
  fe_add(s1, A, B);           // alpha 2
  fe_sub4(E, E, s1);          // alpha 5
  fe_weak(E);                 // tight
  fe_sub(H, B, A);            // alpha 3
  Fe C, D, F, G;
  fe_mul_inl(C, r.T, q.Td);   // 1 x 2
  fe_mul_inl(D, r.Z, q.Z);
  fe_sub(F, D, C);            // alpha 3
  fe_add(G, D, C);            // alpha 2
  fe_mul_inl(r.X, E, F);
  fe_mul_inl(r.Y, G, H);
  fe_mul_inl(r.Z, F, G);
  if (want_t) fe_mul_inl(r.T, E, H);
}

// r = [k]P (+ addend).  On entry r = P (extended, tight); `load_addend(PtExt&)` is only called when has_addend.
// (With CAPY_VB_SYNC every thread of a CUDA block must call this: block barriers then keep the warps on one instruction stream.)
template <int STRIDE, class LoadAddend>
CAPY_HD void pt_var_base_mul(PtExt& r, const Sc& k, uint4* col, bool CONSTANT_TIME, bool has_addend, LoadAddend&& load_addend) {
  uint32_t K[15];
  {
    uint64_t c = 0;
#pragma unroll
    for (int j = 0; j < 14; j++) {
      const uint64_t t = (uint64_t)k.w[j] + 0x88888888u + c;
      K[j] = (uint32_t)t;
      c = t >> 32;
    }
    K[14] = (uint32_t)c;
  }
  vb_store_entry<STRIDE>(col, 0, r);  // 1P
  // iterations 0..6 build 2P..8P, 7..119 are the windows 112..0, 120 adds the addend
  const int n_it = has_addend ? 121 : 120;
#pragma unroll 1
  for (int it = 0; it < n_it; it++) {
    int n_dbl = 0, dgt = 1, store_idx = -1;
    bool do_add = true, ct = false;
    if (it == 0) {
      n_dbl = 1;
      do_add = false;
      store_idx = 1;
    } else if (it < 7) {
      store_idx = it + 1;
    } else if (it < 120) {
      if (it == 7) pt_identity(r);
      else n_dbl = 4;
      dgt = (int)(K[14] & 15u) - (it == 7 ? 0 : 8);
#pragma unroll
      for (int j = 14; j > 0; j--) K[j] = capy_fshl(K[j - 1], K[j], 4);
      K[0] <<= 4;
      ct = CONSTANT_TIME;
    } else {
      PtExt a;  // the table is dead: entry 0 := addend
      load_addend(a);
      vb_store_entry<STRIDE>(col, 0, a);
    }
#pragma unroll 1
    for (int d = 0; d < n_dbl; d++) {
      CAPY_BLOCK_SYNC();  // one instruction stream per block
      vb_double(r, d == n_dbl - 1);
    }
    if (do_add) {
      PtCached e;
      vb_lookup<STRIDE>(e, col, dgt, ct);
      CAPY_BLOCK_SYNC();
      // T is read by the next addition only: while the table is built, and by the addend after the last window
      vb_add(r, e, it < 7 || (it == 119 && has_addend));
    }
    if (store_idx >= 0) vb_store_entry<STRIDE>(col, store_idx, r);
  }
}

}  // namespace capy

// ---- generator and comb-table construction --------------------------------------------------------
namespace capy {

// RFC 8032 Ed448 base point (SURVEY.md App. C.4 item 1), 28-bit limbs
#define CAPY_GX_LIMBS                                                                                           \
  {0x70cc05eu, 0x26a82bcu, 0x0938e26u, 0x80e18b0u, 0x511433bu, 0xf72ab66u, 0x412ae1au, 0xa3d3a46u, 0xa6de324u, \
   0x0f1767eu, 0x4657047u, 0x36da9e1u, 0x5a622bfu, 0xed221d1u, 0x66bed0du, 0x4f1970cu}
#define CAPY_GY_LIMBS                                                                                           \
  {0x230fa14u, 0x08795bfu, 0x7c8ad98u, 0x132c4edu, 0x9c4fdbdu, 0x1ce67c3u, 0x73ad3ffu, 0x05a0c2du, 0x7789c1eu, \
   0xa398408u, 0xa73736cu, 0xc7624beu, 0x03756c9u, 0x2488762u, 0x16eb6bcu, 0x693f467u}

CAPY_HD void pt_generator(PtExt& g) {
  const uint32_t gx[16] = CAPY_GX_LIMBS;
  const uint32_t gy[16] = CAPY_GY_LIMBS;
#pragma unroll
  for (int i = 0; i < 16; i++) {
    g.X.v[i] = gx[i];
    g.Y.v[i] = gy[i];
  }
  fe_one(g.Z);
  fe_mul(g.T, g.X, g.Y);
}

// table entry e := phi(P) as the canonical Niels triple (y' - x', y' + x', 2 d' x' y'), P projective on E:
// P is taken to affine, then pushed through the isogeny
//   phi(x, y) = ( 2xy / (y^2 - x^2),  (y^2 + x^2) / (2 - y^2 - x^2) )     (a homomorphism E -> E')
// The denominators vanish only at points of even order: P must have odd order.
CAPY_HD void fb_niels_entry(uint32_t* e /*[48]*/, const PtExt& acc) {
  Fe zi, x, y, x2, y2, u, v, w, t, xt, yt, two;
  fe_inv(zi, acc.Z);
  fe_mul_call(&x, &acc.X, &zi);
  fe_mul_call(&y, &acc.Y, &zi);
  fe_sqr_call(&x2, &x);
  fe_sqr_call(&y2, &y);
  fe_sub(u, y2, x2);       // y^2 - x^2, alpha 3
  fe_weak(u);
  fe_add(t, y2, x2);       // y^2 + x^2, alpha 2
  fe_zero(two);
  two.v[0] = 2;
  fe_weak(t);
  fe_sub(v, two, t);       // 2 - y^2 - x^2
  fe_weak(v);
  fe_mul_call(&w, &u, &v);
  fe_inv(w, w);            // 1 / (u v)
  fe_mul_call(&xt, &x, &y);
  fe_add(xt, xt, xt);      // 2xy, alpha 2
  fe_weak(xt);
  fe_mul_call(&xt, &xt, &v);
  fe_mul_call(&xt, &xt, &w);  // x' = 2xy / u
  fe_mul_call(&yt, &t, &u);
  fe_mul_call(&yt, &yt, &w);  // y' = (y^2 + x^2) / v
  Fe ymx, ypx, td;
  fe_sub(ymx, yt, xt);
  fe_add(ypx, yt, xt);
  fe_mul_call(&td, &xt, &yt);
  uint64_t R[16];
  for (int k = 0; k < 16; k++) R[k] = (uint64_t)td.v[k] * EDW_2D_TW_ABS;
  Fe td_abs;
  fe_carry_wide(td_abs, R);
  fe_neg(td, td_abs);      // 2 d' x' y' with d' = -39082
  fe_canon(ymx);
  fe_canon(ypx);
  fe_canon(td);
  for (int k = 0; k < 16; k++) {
    e[k] = ymx.v[k];
    e[16 + k] = ypx.v[k];
    e[32 + k] = td.v[k];
  }
}

// table entry e := phi(P) for P = (x, y) given as 112 affine bytes (x || y, little-endian), P of odd order
CAPY_HD void fb_niels_entry_xy(uint32_t* e /*[48]*/, const uint8_t* xy) {
  uint32_t w[14];
  Fe x, y;
  for (int j = 0; j < 14; j++) w[j] = (uint32_t)xy[4 * j] | ((uint32_t)xy[4 * j + 1] << 8) | ((uint32_t)xy[4 * j + 2] << 16) | ((uint32_t)xy[4 * j + 3] << 24);
  fe_from_words(x, w);
  for (int j = 0; j < 14; j++) w[j] = (uint32_t)xy[56 + 4 * j] | ((uint32_t)xy[57 + 4 * j] << 8) | ((uint32_t)xy[58 + 4 * j] << 16) | ((uint32_t)xy[59 + 4 * j] << 24);
  fe_from_words(y, w);
  PtExt p;
  pt_from_affine(p, x, y);
  fb_niels_entry(e, p);
}

// writes the 16 entries of window i of P's comb table: (j+1) * 32^i * phi(P), j < 16.  The multiples are formed on E
// with the complete formulas (5i doublings, then additions of 32^i P).
CAPY_HD void fb_build_window(uint32_t* row /*[16 * 48]*/, int i, const PtExt& p) {
  PtExt base = p;
#pragma unroll 1
  for (int k = 0; k < FB_WBITS * i; k++) pt_double<true>(base, base);
  PtCached cb;
  pt_to_cached(cb, base);
  PtExt acc = base;
#pragma unroll 1
  for (int j = 0; j < FB_ENTRIES; j++) {
    if (j > 0) pt_add_cached<true>(acc, acc, cb);
    fb_niels_entry(row + j * FB_ENTRY_WORDS, acc);
  }
}

// window i of G's comb table
CAPY_HD void fb_build_window(uint32_t* row /*[16 * 48]*/, int i) {
  PtExt g;
  pt_generator(g);
  fb_build_window(row, i, g);
}

}  // namespace capy
