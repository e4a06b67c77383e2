// sponge.cuh -- batched sponge absorb/squeeze with the reference's exact byte layout.
//
// One thread owns one item.  The bytes an item absorbs are never materialised: they are a
// *virtual stream*  P | KB | X | T | pad  that reproduces what the reference builds in a Vec
// before absorbing (SURVEY.md App. B / App. F):
//   P   constant prefix  bytepad(encode_string(N) || encode_string(S), w)   cshake  shake_functions.rs:50-55
//   KB  per-item key block bytepad(encode_string(K), w)                      kmac    shake_functions.rs:80-82
//   X   the message
//   T   trailer: 06|86 (SHA3-d, :25-29, quirk Q2) / 04 (cSHAKE :57) / 00 01 04 (KMACXOF :86 + :57)
//   pad zeros then 0x80, ONLY when the length so far is not a multiple of the rate  sponge.rs:13-15,89-95 (Q1)
// Blocks that lie wholly inside X are loaded straight from global memory (8-byte lanes,
// little-endian = lane value); blocks touching a segment boundary are assembled per lane.
// Absorb = sponge.rs:47-60 (bytes_to_state), squeeze = sponge.rs:25-34 without the wasted
// trailing permutation (quirk Q8).
#pragma once
#include "keccak.cuh"
#include "keccak_pair.cuh"
#include "sponge_job.h"

#ifndef CAPY_SPONGE_MINB
#define CAPY_SPONGE_MINB 3
#endif

namespace capy {

__device__ __forceinline__ uint32_t left_encode_nbytes(uint64_t v) {
  uint32_t nb = 1;
  while (nb < 8 && (v >> (8 * nb)) != 0) nb++;
  return nb;
}

// Loads of message bytes.  COH = true: the bytes were written earlier in the SAME launch by a block on another SM
// (sponge_chain_kernel with a dependent job): they are read from the L2 (ld.global.cg), never from this SM's L1 --
// a line the L1 fetched for the tail of one item may hold stale bytes of the next item's head.
template <bool COH>
__device__ __forceinline__ uint32_t ld_u8(const uint8_t* p) {
  if constexpr (COH) return (uint32_t)__ldcg(p);
  else return (uint32_t)*p;
}
template <bool COH>
__device__ __forceinline__ uint2 ld_lane(const uint2* p) {
  if constexpr (COH) return __ldcg(p);
  else return __ldg(p);
}
template <bool COH>
__device__ __forceinline__ uint32_t ld_word(const uint32_t* p) {
  if constexpr (COH) return __ldcg(p);
  else return __ldg(p);
}

// ---- per-item geometry of the virtual stream  P | KB | X | T | pad --------------------------------------
struct SpongeGeom {
  const uint8_t* prefix;
  uint32_t prefix_len;
  const uint8_t* key;  // nullptr = no key block
  const uint8_t* x;
  uint32_t trailer, hdr_len;
  uint64_t k0, k1;      // key bytes
  uint64_t x0, x1;      // message bytes
  uint64_t t1;          // end of the trailer
  uint64_t p1;          // end of the first pad (quirk Q4 only, else == t1)
  uint64_t padded;      // end of the stream
  uint64_t nblocks;
  bool has_pad1, has_pad;
  uint8_t hdr[12];  // left_encode(w) || left_encode(8 * klen): the head of bytepad(encode_string(K), w)

  // RATE_HINT: the caller's compile-time rate (8 LANES); when the job's rate equals it -- always, except for the 172-byte
  // rate of cSHAKE at D224 (Q7) -- the two divisions by the rate are divisions by a constant
  template <uint32_t RATE_HINT = 0>
  __device__ __forceinline__ void init(const SpongeJob& J, uint64_t i) {
    prefix = J.prefix;
    prefix_len = J.prefix_len;
    key = nullptr;
    uint64_t klen = 0, kb_len = 0;
    hdr_len = 0;
    if (J.keys) {
      if (J.key_off) {
        key = J.keys + J.key_off[i];
        klen = J.key_off[i + 1] - J.key_off[i];
      } else {
        key = J.keys + i * J.key_stride;
        klen = J.key_len;
      }
      const uint32_t w_nb = left_encode_nbytes(J.w), k_nb = left_encode_nbytes(klen * 8);
      const uint64_t content = (uint64_t)(1 + w_nb) + (1 + k_nb) + klen;
      kb_len = (content / J.w + 1) * J.w;  // byte_pad always appends w - len % w zeros (quirk Q3)
      hdr[hdr_len++] = (uint8_t)w_nb;      // aux_functions.rs:11-49
      for (uint32_t q = w_nb; q-- > 0;) hdr[hdr_len++] = (uint8_t)(J.w >> (8 * q));
      hdr[hdr_len++] = (uint8_t)k_nb;
      const uint64_t bits = klen * 8;
      for (uint32_t q = k_nb; q-- > 0;) hdr[hdr_len++] = (uint8_t)(bits >> (8 * q));
    }
    uint64_t xlen;
    if (J.off) {
      x = J.data + J.off[i];
      xlen = J.off[i + 1] - J.off[i];
    } else {
      x = J.data + i * J.msg_stride;
      xlen = J.msg_len;
    }
    trailer = J.trailer;
    if (J.sha3_suffix) trailer = (xlen % 136u == 135u) ? 0x86u : 0x06u;
    k0 = (uint64_t)J.prefix_len + hdr_len;
    k1 = k0 + klen;
    x0 = (uint64_t)J.prefix_len + kb_len;
    x1 = x0 + xlen;
    uint32_t trailer_len = J.trailer_len;
    if (J.q4_rate) {  // shake_functions.rs:59-61 -> :25-29 on the buffer P|X|04
      trailer |= (((x1 + 1) % 136u == 135u) ? 0x86u : 0x06u) << 8;
      trailer_len = 2;
    }
    t1 = x1 + trailer_len;
    // first pad (Q4 only): to a multiple of the SHA3-d rate, only when unaligned
    p1 = t1;
    has_pad1 = false;
    if (J.q4_rate) {
      const uint64_t rem1 = t1 % J.q4_rate;
      has_pad1 = rem1 != 0;
      if (has_pad1) p1 = t1 + (J.q4_rate - rem1);
    }
    uint64_t rem;
    if (RATE_HINT != 0 && J.rate == RATE_HINT) {
      rem = p1 % RATE_HINT;
      padded = rem ? p1 + (RATE_HINT - rem) : p1;  // Q1: no pad block when aligned
      nblocks = padded / RATE_HINT;
    } else {
      rem = p1 % J.rate;
      padded = rem ? p1 + (J.rate - rem) : p1;
      nblocks = padded / J.rate;
    }
    has_pad = rem != 0;
    if (J.fips_pad && !has_pad) trailer |= 0x80u << (8 * (trailer_len - 1));
  }

  // The stream of a resumable item (SpongeResume): the carry stands in the place of P, so this job absorbs  carry | X  (an
  // update: whole blocks only, no trailer, no pad) or  carry | T | pad  (the final job).  Everything before the carry was
  // block-aligned, so the carry and T alone decide whether there is a pad block (Q1), and the SHA3-d suffix comes from
  // the total length (Q2).  RATE is lane-aligned: D224 KMAC (Q7) is not resumable.
  template <uint32_t RATE>
  __device__ __forceinline__ void init_resume(const SpongeJob& J, const SpongeResume& R, uint64_t i) {
    const uint64_t total = R.totals[i];
    const bool update = J.chain_out != nullptr;
    prefix = R.carry + i * RATE;
    prefix_len = (uint32_t)(total % RATE);
    key = nullptr;
    hdr_len = 0;
    k0 = k1 = x0 = prefix_len;
    x = prefix;
    uint64_t xlen = 0;
    if (update) {
      x = J.data + J.off[i];
      xlen = J.off[i + 1] - J.off[i];
    }
    x1 = x0 + xlen;
    trailer = update ? 0u : J.sha3_suffix ? ((total % 136u == 135u) ? 0x86u : 0x06u) : J.trailer;
    t1 = p1 = x1 + (update ? 0u : J.trailer_len);
    has_pad1 = false;
    const uint64_t rem = t1 % RATE;
    has_pad = !update && rem != 0;
    padded = has_pad ? t1 + (RATE - rem) : t1;
    nblocks = padded / RATE;  // an update: the whole blocks of carry | X
  }

  // bytes of the segment [seg0, seg1) (stream offsets; base[0] sits at seg0) that fall into the lane at o
  template <bool COH = false>
  static __device__ __forceinline__ uint64_t piece(const uint8_t* base, uint64_t seg0, uint64_t seg1, uint64_t o) {
    const uint64_t lo = o > seg0 ? o : seg0, hi = o + 8 < seg1 ? o + 8 : seg1;
    uint64_t v = 0;
#pragma unroll 1
    for (uint64_t q = lo; q < hi; q++) v |= (uint64_t)ld_u8<COH>(base + (q - seg0)) << (8 * (uint32_t)(q - o));
    return v;
  }

  // The 8-byte lane at stream offset o of a boundary block: the OR of the pieces of the (at most five) segments
  // that overlap it, each piece fetched with a loop over just its own bytes; lanes wholly inside X, inside zero
  // padding or past the end take one compare each.  (The first version walked all 8 bytes of every lane through
  // a compare chain: ~2 700 instructions per block against ~700 now; KMAC over 4 KB has two such blocks in 33.)
  template <bool COH = false>
  __device__ __forceinline__ uint64_t lane(uint64_t o) const {
    uint64_t v = 0;
    if (o >= x0 && o + 8 <= x1) {
      const uint8_t* p = x + (o - x0);
#pragma unroll
      for (int k = 0; k < 8; k++) v |= (uint64_t)ld_u8<COH>(p + k) << (8 * k);
    } else if (o < padded && !(o >= k1 && o + 8 <= x0) && !(o >= t1 && o + 8 < p1) && !(o >= p1 && o + 8 < padded)) {
      if (o < prefix_len) v |= piece(prefix, 0, prefix_len, o);
      if (key && o + 8 > prefix_len && o < k1) {
        v |= piece(hdr, prefix_len, k0, o);
        v |= piece(key, k0, k1, o);
      }
      if (o + 8 > x0 && o < x1) v |= piece<COH>(x, x0, x1, o);
      if (o + 8 > x1 && o < t1) v |= x1 >= o ? (uint64_t)trailer << (8 * (uint32_t)(x1 - o)) : (uint64_t)trailer >> (8 * (uint32_t)(o - x1));
      if (has_pad1 && p1 - 1 >= o && p1 - 1 < o + 8) v |= 0x80ull << (8 * (uint32_t)(p1 - 1 - o));
      if (has_pad && padded - 1 >= o && padded - 1 < o + 8) v |= 0x80ull << (8 * (uint32_t)(padded - 1 - o));
    }
    return v;
  }

  // blocks [fb0, fb1) lie wholly inside X (stride = bytes consumed per block)
  __device__ __forceinline__ void fast_range(uint64_t stride, uint64_t skip_blocks, uint64_t& fb0, uint64_t& fb1) const {
    fb0 = (x0 + stride - 1) / stride;
    fb1 = x1 / stride;
    if (fb0 < skip_blocks) fb0 = skip_blocks;
    if (fb1 > nblocks) fb1 = nblocks;
    if (fb1 < fb0) fb1 = fb0;
    if (fb0 > nblocks) fb0 = fb1 = nblocks;
  }
};

// =====================================================================================================
// one thread per item
// =====================================================================================================
// CHAIN: the item may start from / stop at a handed-over state (rank = its slot in the hand-off arrays); the plain
// kernels instantiate CHAIN = false and compile to what they were.
// COH: the message was written earlier in this launch (dependent job): see ld_u8.
// RESUME (with CHAIN): the item is the resumable stream R describes (SpongeGeom::init_resume); an update also leaves the
// new carry and total behind.
template <int LANES, bool CHAIN = false, bool COH = false, bool RESUME = false>
__device__ __forceinline__ void sponge_item(const SpongeJob& J, uint64_t i, uint64_t rank = 0, const SpongeResume* R = nullptr) {
  SpongeGeom g;
  uint64_t state_n = J.n;
  if constexpr (RESUME) {
    g.template init_resume<8u * LANES>(J, *R, i);
    state_n = R->state_n;
  }
  else g.template init<8u * LANES>(J, i);
  Lane a[25];
  if (CHAIN && J.chain_in) {
#pragma unroll
    for (int k = 0; k < 25; k++) {
      const uint64_t v = __ldcg(J.chain_in + (uint64_t)k * state_n + rank);  // written by another SM in this launch: L2, not L1
      a[k].lo = (uint32_t)v;
      a[k].hi = (uint32_t)(v >> 32);
    }
  } else if (J.init_state) {
#pragma unroll
    for (int k = 0; k < 25; k++) {
      const uint64_t v = J.init_state[k];
      a[k].lo = (uint32_t)v;
      a[k].hi = (uint32_t)(v >> 32);
    }
  } else {
    state_zero(a);
  }

  // ---- absorb (sponge.rs:47-60) -------------------------------------------------------
  // Blocks [fb0, fb1) lie wholly inside X: they are loaded straight from global memory, with the next
  // block's loads issued BEFORE the current permutation (software prefetch: at one warp per scheduler --
  // the long-message launch -- there is no other warp to hide the load latency).  The blocks before and
  // after that range touch a segment boundary and are assembled lane by lane from the virtual stream.
  constexpr uint64_t STRIDE = 8ull * LANES;  // bytes consumed per block (168 for the 172 quirk)
  uint64_t fb0, fb1;
  g.fast_range(STRIDE, J.skip_blocks, fb0, fb1);
  uint64_t nblocks = g.nblocks;
  if (CHAIN && J.chain_out) {  // this segment ends at stop_block
    nblocks = nblocks < J.stop_block ? nblocks : J.stop_block;
    fb0 = fb0 < nblocks ? fb0 : nblocks;
    fb1 = fb1 < nblocks ? fb1 : nblocks;
  }

  auto slow_block = [&](uint64_t b) {
    const uint64_t s = b * STRIDE;
    uint64_t blk[LANES];
#pragma unroll 1
    for (int j = 0; j < LANES; j++) blk[j] = g.template lane<COH>(s + 8ull * j);
#pragma unroll
    for (int j = 0; j < LANES; j++) {
      a[j].lo ^= (uint32_t)blk[j];
      a[j].hi ^= (uint32_t)(blk[j] >> 32);
    }
    keccak_f1600(a);
  };

#pragma unroll 1
  for (uint64_t b = J.skip_blocks; b < fb0; b++) slow_block(b);

  // The choice between the 8-byte-aligned and the byte-phase load path is made PER WARP: a per-thread
  // branch here would put two separate permutation loops on the two sides of a divergent branch and
  // the warp would run both back to back (measured 2.1x slower on ragged batches).
  const uint8_t* p = g.x + (fb0 * STRIDE - g.x0);
  const bool has_fast = fb0 < fb1;
  const bool my_aligned = !has_fast || (reinterpret_cast<uintptr_t>(p) & 7u) == 0;
#if defined(__CUDA_ARCH__)
  const bool warp_aligned = __all_sync(__activemask(), my_aligned);
#else
  const bool warp_aligned = my_aligned;
#endif
  if (warp_aligned) {
    const uint2* q = reinterpret_cast<const uint2*>(p);
    uint2 cur[LANES];
    if (has_fast) {
#pragma unroll
      for (int j = 0; j < LANES; j++) cur[j] = ld_lane<COH>(q + j);
    }
#pragma unroll 1
    for (uint64_t b = fb0; b < fb1; b++) {
      q += LANES;
      uint2 nxt[LANES];
      if (b + 1 < fb1) {  // (as predicated loads, the way the pair tier has them, this loop measured 1 % slower)
#pragma unroll
        for (int j = 0; j < LANES; j++) nxt[j] = ld_lane<COH>(q + j);
      }
#pragma unroll
      for (int j = 0; j < LANES; j++) {
        a[j].lo ^= cur[j].x;
        a[j].hi ^= cur[j].y;
      }
      keccak_f1600(a);
#pragma unroll
      for (int j = 0; j < LANES; j++) cur[j] = nxt[j];
    }
  } else {
    // any byte phase: aligned 32-bit words + funnel shift (sh == 0 for 4-byte aligned starts)
    const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3u) * 8u;
    const uint32_t* q = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
    uint32_t cw[2 * LANES + 1];
    if (has_fast) {
#pragma unroll
      for (int j = 0; j < 2 * LANES; j++) cw[j] = ld_word<COH>(q + j);
      // the last word is only needed (and only guaranteed readable) when sh != 0
      cw[2 * LANES] = sh != 0 ? ld_word<COH>(q + 2 * LANES) : 0u;
    }
#pragma unroll 1
    for (uint64_t b = fb0; b < fb1; b++) {
      q += 2 * LANES;
      uint32_t nw[2 * LANES + 1];
      if (b + 1 < fb1) {
#pragma unroll
        for (int j = 0; j < 2 * LANES; j++) nw[j] = ld_word<COH>(q + j);
        nw[2 * LANES] = sh != 0 ? ld_word<COH>(q + 2 * LANES) : 0u;
      }
#pragma unroll
      for (int j = 0; j < LANES; j++) {
        a[j].lo ^= __funnelshift_r(cw[2 * j], cw[2 * j + 1], sh);
        a[j].hi ^= __funnelshift_r(cw[2 * j + 1], cw[2 * j + 2], sh);
      }
      keccak_f1600(a);
#pragma unroll
      for (int j = 0; j < 2 * LANES + 1; j++) cw[j] = nw[j];
    }
  }

  // The stream usually ends with exactly one block "message tail | trailer | zeros | 0x80" that starts inside (or at the
  // end of) the message, and short messages ARE that block.  It is assembled from aligned 32-bit words + funnel shift like
  // the whole-message blocks (only words that hold a message byte are read), the bytes behind the message masked away:
  // ~250 instructions instead of the ~2 500 of the general lane-by-lane assembly.  2^20 ragged messages of 1..135 bytes
  // through capy_sha3_batch_dev: 0.52 -> 0.32 ms (profiles/README.md, r02c).  Not for the Q4 double padding, a rate that
  // is not a whole number of lanes (Q7 at D224), or a trailer that spills into a second block: those take the general path.
  const bool simple_tail = !(CHAIN && J.chain_out) && J.q4_rate == 0 && J.rate == (uint32_t)STRIDE && fb1 + 1 == nblocks &&
                           fb1 * STRIDE >= g.x0 && fb1 * STRIDE <= g.x1 && fb1 >= J.skip_blocks;
  if (simple_tail) {
    const uint64_t s0 = fb1 * STRIDE;
    const uint32_t rem = (uint32_t)(g.x1 - s0);  // message bytes in this block: 0 .. STRIDE - 1
    const uint8_t* tp = g.x + (s0 - g.x0);
    const uint32_t ph = (uint32_t)(reinterpret_cast<uintptr_t>(tp) & 3u), tsh = 8u * ph;
    const uint32_t* tq = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(tp) & ~(uintptr_t)3);
    const uint32_t nw = rem ? (rem + ph + 3u) / 4u : 0u;  // words that hold at least one message byte
    uint32_t w[2 * LANES + 1];
#pragma unroll
    for (int j = 0; j < 2 * LANES + 1; j++) {
      w[j] = 0u;
      if ((uint32_t)j < nw) w[j] = ld_word<COH>(tq + j);
    }
    const uint64_t tr = g.trailer;  // up to three bytes (KMACXOF: 00 01 04), little-endian
#pragma unroll
    for (int j = 0; j < LANES; j++) {
      uint32_t lo = __funnelshift_r(w[2 * j], w[2 * j + 1], tsh), hi = __funnelshift_r(w[2 * j + 1], w[2 * j + 2], tsh);
      const uint32_t o = 8u * j;
      // keep the message bytes below rem, put the trailer bytes at rem ..
      const uint32_t klo = rem > o ? (rem - o >= 4u ? 0xffffffffu : (1u << (8u * (rem - o))) - 1u) : 0u;
      const uint32_t khi = rem > o + 4u ? (rem - o - 4u >= 4u ? 0xffffffffu : (1u << (8u * (rem - o - 4u))) - 1u) : 0u;
      lo &= klo;
      hi &= khi;
      if (rem + 4u > o && rem < o + 8u) {
        const uint64_t t = rem >= o ? tr << (8u * (rem - o)) : tr >> (8u * (o - rem));
        lo |= (uint32_t)t;
        hi |= (uint32_t)(t >> 32);
      }
      a[j].lo ^= lo;
      a[j].hi ^= hi;
    }
    if (g.has_pad) a[LANES - 1].hi ^= 0x80000000u;  // (Q1: no 0x80 when the trailer filled the block exactly)
    keccak_f1600(a);
  } else {
#pragma unroll 1
    for (uint64_t b = fb1; b < nblocks; b++) slow_block(b);
  }

  if (CHAIN && J.chain_out) {  // hand the state to the next segment (coalesced: lane k of rank r at [k * n + r])
#pragma unroll
    for (int k = 0; k < 25; k++) J.chain_out[(uint64_t)k * state_n + rank] = ((uint64_t)a[k].hi << 32) | a[k].lo;
    if constexpr (RESUME) {  // an update: the bytes behind the last whole block are the new carry (the old one was read above)
      uint8_t* cb = R->carry + i * STRIDE;
      const uint64_t s0 = nblocks * STRIDE;
#pragma unroll 1
      for (uint64_t q = s0 > g.x0 ? s0 : g.x0; q < g.x1; q++) cb[q - s0] = g.x[q - g.x0];
      R->totals[i] += g.x1 - g.x0;
    }
    return;
  }

  // ---- squeeze (sponge.rs:25-34, minus the dropped final permutation) -----------------------
  uint8_t* o;
  uint64_t out_bytes;
  if (J.out_off) {
    o = J.out + J.out_off[i];
    out_bytes = J.out_off[i + 1] - J.out_off[i];
  } else {
    o = J.out + i * J.out_stride;
    out_bytes = J.out_bytes;
  }
  const uint64_t sq_bytes = 8ull * J.sq_lanes;
  const uint8_t* xi = J.xor_in ? J.xor_in + (o - J.out) : nullptr;
  const bool o_aligned = (reinterpret_cast<uintptr_t>(o) & 7u) == 0 && (!xi || (reinterpret_cast<uintptr_t>(xi) & 7u) == 0);
  // keystream shape (out = squeeze ^ xor_in, sha3/encryptable.rs:41-42) with whole aligned blocks of LANES lanes: the
  // words of xor_in for the NEXT block are loaded before the permutation, like the absorb loop does with the message
  // (the loads of a block used to sit right in front of the XOR that needs them: long_scoreboard 0.52 in the seal).
  const bool xor_pipelined = xi && o_aligned && (int)J.sq_lanes == LANES;
  uint2 xm[LANES];
  if (xor_pipelined && sq_bytes <= out_bytes) {
#pragma unroll
    for (int j = 0; j < LANES; j++) xm[j] = reinterpret_cast<const uint2*>(xi)[j];
  }
  for (uint64_t produced = 0; produced < out_bytes;) {
    if (o_aligned && produced + sq_bytes <= out_bytes) {
      // whole squeeze block, 8-byte aligned: straight stores (the keystream / long-output shape)
      uint2* op = reinterpret_cast<uint2*>(o + produced);
      if (xor_pipelined) {
#pragma unroll
        for (int j = 0; j < LANES; j++) op[j] = make_uint2(a[j].lo ^ xm[j].x, a[j].hi ^ xm[j].y);
        produced += sq_bytes;
        if (produced + sq_bytes <= out_bytes) {
          const uint2* xp = reinterpret_cast<const uint2*>(xi + produced);
#pragma unroll
          for (int j = 0; j < LANES; j++) xm[j] = xp[j];
        }
        if (produced < out_bytes) keccak_f1600(a);
        continue;
      }
      const uint2* xp = reinterpret_cast<const uint2*>(xi ? xi + produced : nullptr);
#pragma unroll
      for (int j = 0; j < 21; j++) {
        if (j < (int)J.sq_lanes) {
          uint2 v = make_uint2(a[j].lo, a[j].hi);
          if (xi) {
            const uint2 m = xp[j];
            v.x ^= m.x;
            v.y ^= m.y;
          }
          op[j] = v;
        }
      }
      produced += sq_bytes;
      if (produced < out_bytes) keccak_f1600(a);
      continue;
    }
#pragma unroll
    for (int j = 0; j < 21; j++) {
      const uint64_t pos = produced + 8ull * j;
      if (j < (int)J.sq_lanes && pos < out_bytes) {
        if (o_aligned && pos + 8 <= out_bytes) {
          uint2 v = make_uint2(a[j].lo, a[j].hi);
          if (xi) {
            const uint2 m = *reinterpret_cast<const uint2*>(xi + pos);
            v.x ^= m.x;
            v.y ^= m.y;
          }
          *reinterpret_cast<uint2*>(o + pos) = v;
        } else {
          const uint64_t v = ((uint64_t)a[j].hi << 32) | a[j].lo;
          for (int k = 0; k < 8 && pos + k < out_bytes; k++)
            o[pos + k] = (uint8_t)(v >> (8 * k)) ^ (xi ? xi[pos + k] : (uint8_t)0);
        }
      }
    }
    produced += sq_bytes;
    if (produced < out_bytes) keccak_f1600(a);
  }
}

// =====================================================================================================
// two threads per item (keccak_pair.cuh): the even thread holds the low, the odd thread the high 32 bits of
// every lane.  The permutation exchanges halves with full-warp shuffles, so the sixteen pairs of a warp walk ONE
// warp-uniform step loop: step s of an item is "absorb block s", then "emit squeeze block s - absorbed", and every
// step ends in a permutation that all 32 threads execute together; items that are already finished (the batch
// is length-sorted, so the spread inside a warp is small) keep permuting a state nobody reads any more.
// =====================================================================================================
// The rare paths of the fast tiers live out of line.  Inlined, their byte loads and stores shared scoreboards with the
// prefetch loads of the hot path: the first instruction of the permutation sits behind the point where all paths of a step
// meet, and there the compiler waited for "the scoreboard" -- i.e. for the loads of the NEXT block that had just been
// issued (ncu: 15 % of all stall samples of the pair tier on that one instruction, long scoreboard).  A call returns with
// nothing in flight.  (The squeeze-block emit of the pair tier stays inline: out of line it measured 2 % slower.)
__device__ __noinline__ uint64_t sponge_lane_ool(const SpongeGeom* g, uint64_t o) { return g->lane(o); }

template <int LANES>
__device__ __forceinline__ void sponge_item_pair(const SpongeJob& J, uint64_t i, bool valid, uint32_t half) {
  constexpr uint64_t STRIDE = 8ull * LANES;
  SpongeGeom g;
  uint64_t fb0 = 0, fb1 = 0, n_absorb = 0, n_steps = 0;
  uint8_t* o = nullptr;
  const uint8_t* xi = nullptr;
  uint64_t out_bytes = 0;
  const uint32_t sq_lanes = J.sq_lanes;  // (J lives in memory behind a reference: keep what the step loop needs in registers)
  const uint64_t skip = J.skip_blocks;
  const uint64_t sq_bytes = 8ull * sq_lanes;
  if (valid) {
    g.init(J, i);
    g.fast_range(STRIDE, skip, fb0, fb1);
    n_absorb = g.nblocks - skip;
    if (J.out_off) {
      o = J.out + J.out_off[i];
      out_bytes = J.out_off[i + 1] - J.out_off[i];
    } else {
      o = J.out + i * J.out_stride;
      out_bytes = J.out_bytes;
    }
    xi = J.xor_in ? J.xor_in + (o - J.out) : nullptr;
    // absorb steps, then one step per squeeze block except the last (no permutation follows it, quirk Q8)
    n_steps = n_absorb + (out_bytes ? (out_bytes + sq_bytes - 1) / sq_bytes - 1 : 0);
  }
  const bool o_aligned = (reinterpret_cast<uintptr_t>(o) & 3u) == 0 && (!xi || (reinterpret_cast<uintptr_t>(xi) & 3u) == 0);
  // warp-uniform trip count (64-bit maximum over the warp from two 32-bit reductions)
  const uint32_t hi_max = __reduce_max_sync(0xffffffffu, (uint32_t)(n_steps >> 32));
  const uint32_t lo_max = __reduce_max_sync(0xffffffffu, (uint32_t)(n_steps >> 32) == hi_max ? (uint32_t)n_steps : 0u);
  const uint64_t warp_steps = ((uint64_t)hi_max << 32) | lo_max;

  uint32_t h[25];
#pragma unroll
  for (int k = 0; k < 25; k++) h[k] = J.init_state ? (half ? (uint32_t)(J.init_state[k] >> 32) : (uint32_t)J.init_state[k]) : 0u;

  // each thread streams only its own 32-bit half of every lane of the whole-message blocks; any byte phase:
  // aligned words + funnel shift, next block prefetched before the permutation
  const uint8_t* p = valid ? g.x + (fb0 * STRIDE - g.x0) : nullptr;
  const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3u) * 8u;
  const uint32_t* q = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3) + half;
  uint32_t c0[LANES], c1[LANES];
#pragma unroll
  for (int j = 0; j < LANES; j++) c0[j] = c1[j] = 0u;
  if (fb0 < fb1) {
#pragma unroll
    for (int j = 0; j < LANES; j++) {
      c0[j] = __ldg(q + 2 * j);
      c1[j] = sh != 0 ? __ldg(q + 2 * j + 1) : 0u;
    }
  }

  auto emit = [&](uint64_t sb) {  // squeeze block sb of this item (sponge.rs:25-34)
    const uint64_t produced = sb * sq_bytes;
#pragma unroll
    for (int j = 0; j < 21; j++) {
      const uint64_t hp = produced + 8ull * j + 4ull * half;  // this thread's four bytes of lane j
      if (j < (int)sq_lanes && hp < out_bytes) {
        if (o_aligned && hp + 4 <= out_bytes) {
          uint32_t v = h[j];
          if (xi) v ^= *reinterpret_cast<const uint32_t*>(xi + hp);
          *reinterpret_cast<uint32_t*>(o + hp) = v;
        } else {
          for (int k = 0; k < 4 && hp + k < out_bytes; k++) o[hp + k] = (uint8_t)(h[j] >> (8 * k)) ^ (xi ? xi[hp + k] : (uint8_t)0);
        }
      }
    }
  };

#pragma unroll 1
  for (uint64_t s = 0; s <= warp_steps; s++) {
    bool pf = false;  // fetch the next whole-message block (below, behind the point where the paths of a step meet)
    if (s < n_absorb) {
      const uint64_t b = skip + s;
      if (b >= fb0 && b < fb1) {
#pragma unroll
        for (int j = 0; j < LANES; j++) h[j] ^= __funnelshift_r(c0[j], c1[j], sh);
        q += 2 * LANES;
        pf = b + 1 < fb1;
      } else {
        uint32_t blk[LANES];
#pragma unroll 1
        for (int j = 0; j < LANES; j++) {
          const uint64_t v = sponge_lane_ool(&g, b * STRIDE + 8ull * j);
          blk[j] = half ? (uint32_t)(v >> 32) : (uint32_t)v;
        }
#pragma unroll
        for (int j = 0; j < LANES; j++) h[j] ^= blk[j];
      }
    } else if (s <= n_steps && out_bytes) {
      emit(s - n_absorb);
    }
    // The loads of the next block are issued HERE, as predicated loads on the straight line into the permutation.  Inside
    // the absorb branch they sat in front of the point where the paths of a step meet, and the first instruction of the
    // permutation waited there for the scoreboard they share with the rare paths -- i.e. for the loads just issued
    // (ncu: 15 % of the pair tier's stall samples on that one instruction, long scoreboard).
    const bool pf1 = pf && sh != 0;
#pragma unroll
    for (int j = 0; j < LANES; j++) {
      if (pf) c0[j] = __ldg(q + 2 * j);
      if (pf1) c1[j] = __ldg(q + 2 * j + 1);
    }
    if (s < warp_steps) keccak_f1600_pair(h, half);
  }
}

// =====================================================================================================
// one WARP per item (WarpKeccak): thread l owns lane l, absorbs its own 8 bytes of every block (a warp reads one
// message as contiguous 72..168-byte rows) and emits its own lane of every squeeze block
// =====================================================================================================
template <int LANES>
__device__ __noinline__ void sponge_item_warp(const SpongeJob& J, uint64_t i) {  // own register allocation: fused inline it slowed the other tiers
  constexpr uint64_t STRIDE = 8ull * LANES;
  const int l = threadIdx.x & 31;
  const bool mine = l < LANES;
  SpongeGeom g;
  g.init(J, i);
  uint64_t fb0, fb1;
  g.fast_range(STRIDE, J.skip_blocks, fb0, fb1);
  WarpKeccak wk;
  wk.init(l);
  uint32_t lo = 0, hi = 0;
  if (J.init_state && l < 25) {
    const uint64_t v = J.init_state[l];
    lo = (uint32_t)v;
    hi = (uint32_t)(v >> 32);
  }
  // whole-message blocks: this thread's lane as three aligned words + funnel shift, next block prefetched.  Threads
  // beyond the rate shadow lane 0 and mask their value away, so the hot loop has no divergent branch in front of the
  // full-warp shuffles.
  const uint32_t keep = mine ? 0xffffffffu : 0u;
  const uint8_t* p = g.x + (fb0 * STRIDE - g.x0) + 8ull * (mine ? l : 0);
  const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3u) * 8u;
  const uint32_t* q = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
  uint32_t w0 = 0, w1 = 0, w2 = 0;
  if (fb0 < fb1) {
    w0 = __ldg(q);
    w1 = __ldg(q + 1);
    w2 = sh != 0 ? __ldg(q + 2) : 0u;
  }
  const uint64_t nblocks = g.nblocks, skip = J.skip_blocks;
#pragma unroll 1
  for (uint64_t b = skip; b < nblocks; b++) {
    uint32_t vlo, vhi;
    bool pf = false;
    if (b >= fb0 && b < fb1) {  // warp-uniform: one item per warp
      vlo = __funnelshift_r(w0, w1, sh);
      vhi = __funnelshift_r(w1, w2, sh);
      q += 2 * LANES;
      pf = b + 1 < fb1;
    } else {
      const uint64_t v = sponge_lane_ool(&g, b * STRIDE + 8ull * (mine ? l : 0));
      vlo = (uint32_t)v;
      vhi = (uint32_t)(v >> 32);
    }
    lo ^= vlo & keep;
    hi ^= vhi & keep;
    // next block: predicated loads behind the point where the two paths meet (see sponge_item_pair)
    if (pf) w0 = __ldg(q);
    if (pf) w1 = __ldg(q + 1);
    if (pf && sh != 0) w2 = __ldg(q + 2);
    wk.permute(lo, hi);
  }
  // squeeze (sponge.rs:25-34, minus the dropped final permutation)
  uint8_t* o;
  uint64_t out_bytes;
  if (J.out_off) {
    o = J.out + J.out_off[i];
    out_bytes = J.out_off[i + 1] - J.out_off[i];
  } else {
    o = J.out + i * J.out_stride;
    out_bytes = J.out_bytes;
  }
  const uint64_t sq_bytes = 8ull * J.sq_lanes;
  const uint8_t* xi = J.xor_in ? J.xor_in + (o - J.out) : nullptr;
  const bool o_aligned = (reinterpret_cast<uintptr_t>(o) & 7u) == 0 && (!xi || (reinterpret_cast<uintptr_t>(xi) & 7u) == 0);
#pragma unroll 1
  for (uint64_t produced = 0; produced < out_bytes;) {
    const uint64_t pos = produced + 8ull * l;
    if (l < (int)J.sq_lanes && pos < out_bytes) {
      if (o_aligned && pos + 8 <= out_bytes) {
        uint2 v = make_uint2(lo, hi);
        if (xi) {
          const uint2 mm = *reinterpret_cast<const uint2*>(xi + pos);
          v.x ^= mm.x;
          v.y ^= mm.y;
        }
        *reinterpret_cast<uint2*>(o + pos) = v;
      } else {
        const uint64_t v = ((uint64_t)hi << 32) | lo;
        for (int k = 0; k < 8 && pos + k < out_bytes; k++) o[pos + k] = (uint8_t)(v >> (8 * k)) ^ (xi ? xi[pos + k] : (uint8_t)0);
      }
    }
    produced += sq_bytes;
    if (produced < out_bytes) wk.permute(lo, hi);
  }
}

// rank r of the (length-sorted) work list -> item index
__device__ __forceinline__ uint64_t sponge_rank_item(const SpongeJob& J, uint64_t r) { return J.order ? (uint64_t)J.order[r] : r; }

// one thread per item: ranks [J.first, J.n)
template <int LANES>
__global__ void __launch_bounds__(128, CAPY_SPONGE_MINB) sponge_kernel(const SpongeJob J) {
  const uint64_t r = J.first + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= J.n) return;
  sponge_item<LANES>(J, sponge_rank_item(J, r));
}

// Two jobs over the same number of items in one launch: warps alternate between job 0 and job 1 (warp w works on
// job w & 1, ranks 32 (w >> 1) ..), so neither job waits for the other's blocks and no warp mixes the two code paths.
struct SpongeJob2 {
  SpongeJob j[2];
};
template <int LANES>
__global__ void __launch_bounds__(128, CAPY_SPONGE_MINB) sponge_kernel2(const __grid_constant__ SpongeJob2 JJ) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const SpongeJob& J = JJ.j[(t >> 5) & 1u];
  const uint64_t r = ((t >> 6) << 5) | (t & 31u);
  if (r >= J.n) return;
  sponge_item<LANES>(J, sponge_rank_item(J, r));
}

// A uniform batch whose warps fill the schedulers unevenly (2^16 items = 3.46 warps per scheduler: a quarter of the
// schedulers carry a fourth warp and everybody waits for them) is cut in two along the chains: job 0 absorbs the first
// half of every item's blocks and stores the state, job 1 picks the states up and finishes.  Twice the warps, half as long
// each: 6.92 per scheduler.  Both jobs are ONE launch; a block takes a ticket when it starts, the first `blocks_per_job`
// tickets work on job 0, the others on job 1, and a job-1 block waits for the job-0 block of the same items (which holds a
// smaller ticket, so it is running or done: no deadlock).  The launcher only cuts batches with at least as many job-0
// blocks as the GPU holds at once, so in practice nobody waits.  A launch of only `blocks_per_job` blocks runs job 0 alone
// (every ticket is a job-0 ticket, nobody waits): the updates and finals of resumable streams (SpongeResume).  An update
// of encryption streams runs both jobs at any size -- the tag stream's update, then its keystream (SpongeSqueeze) -- and
// its job-1 blocks wait only for job-0 blocks that took their tickets earlier.
struct SpongeChain {
  SpongeJob j[2];
  uint32_t* sync;  // [0] ticket counter, [1 + b] warps of job-0 block b that have stored their states; zeroed before the launch
  uint32_t blocks_per_job;
  // job 1 reads, as its message, bytes that job 0 wrote for the same item (the two passes of an authenticated
  // decryption: keystream XOR, then the tag over the plaintext): its message loads go to the L2
  uint32_t data_dependent;
  SpongeResume resume;  // carry == nullptr: the jobs are not resumable streams
  SpongeSqueeze squeeze;  // resumable streams with two jobs: job 1 is the keystream update of encryption streams
  SpongeDual dual;        // b_state != nullptr: job 0 runs two states in lockstep (sign and decryption streams)
};
// resumable streams (order == nullptr: rank = item), out of line: the cut chains keep their own register allocation
template <int LANES>
__device__ __noinline__ void sponge_item_resume_ool(const SpongeJob& J, const SpongeResume* R, uint64_t i) {
  sponge_item<LANES, true, false, true>(J, i, i, R);
}

// Keystream update of item i (SpongeSqueeze): squeeze blocks of 8 LANES bytes (the cSHAKE / KMAC squeeze width equals the
// rate at D256 / 384 / 512), entered at any byte of a block.  Lane j of a block is keystream bytes [8 j, 8 j + 8) of it; a
// lane wholly inside the piece is one 8-byte load and store when data and out put keystream lanes on 8-byte boundaries
// (pieces whose offsets and positions agree mod 8: the usual packed batch), any other lane goes byte by byte.  Out of line
// like the resume path.
template <int LANES>
__device__ __noinline__ void sponge_squeeze_resume_ool(const SpongeJob& J, const SpongeSqueeze* S, uint64_t i) {
  constexpr uint64_t SQ = 8ull * LANES;
  const uint64_t state_n = S->state_n;
  Lane a[25];
#pragma unroll
  for (int k = 0; k < 25; k++) {
    const uint64_t v = J.chain_in[(uint64_t)k * state_n + i];
    a[k].lo = (uint32_t)v;
    a[k].hi = (uint32_t)(v >> 32);
  }
  const uint64_t p0 = S->pos[i], a0 = J.off[i], p1 = p0 + (J.off[i + 1] - a0);
  const uint8_t* x = J.data + a0;  // keystream byte p goes with x[p - p0] and o[p - p0]
  uint8_t* o = J.out + a0;
  const bool al = ((reinterpret_cast<uintptr_t>(x) - p0) & 7u) == 0 && ((reinterpret_cast<uintptr_t>(o) - p0) & 7u) == 0;
#pragma unroll 1
  for (uint64_t b = p0 - p0 % SQ; b < p1;) {
#pragma unroll
    for (int j = 0; j < LANES; j++) {
      const uint64_t l0 = b + 8ull * j, lo = l0 > p0 ? l0 : p0, hi = l0 + 8 < p1 ? l0 + 8 : p1;
      if (lo < hi) {
        if (al && hi - lo == 8) {
          const uint2 m = *reinterpret_cast<const uint2*>(x + (lo - p0));
          *reinterpret_cast<uint2*>(o + (lo - p0)) = make_uint2(a[j].lo ^ m.x, a[j].hi ^ m.y);
        } else {
          const uint64_t v = ((uint64_t)a[j].hi << 32) | a[j].lo;
#pragma unroll 1
          for (uint64_t q = lo; q < hi; q++) o[q - p0] = x[q - p0] ^ (uint8_t)(v >> (8 * (uint32_t)(q - l0)));
        }
      }
    }
    b += SQ;
    if (b <= p1) keccak_f1600(a);  // this block is used up: the next byte comes from the next one
  }
#pragma unroll
  for (int k = 0; k < 25; k++) J.chain_out[(uint64_t)k * state_n + i] = ((uint64_t)a[k].hi << 32) | a[k].lo;
  S->pos[i] = p1;
}

// Two states of item i in lockstep (SpongeDual), entered at any byte of a block.  Block s of the stream is carry | piece
// bytes; a block that the piece completes goes into B (and into A in dual absorb) and both states permute, the bytes of
// an incomplete last block join the carry.  Lanes wholly inside the piece take the 8-byte path of
// sponge_squeeze_resume_ool, any other lane goes byte by byte.  In the open mode the plaintext exists only in registers,
// in the stream's own carry and in `out`: fused, because the tag depends on the keystream output, and two jobs would have
// to pass the unverified plaintext through a buffer the stream does not own.
template <int LANES>
__device__ __noinline__ void sponge_dual_resume_ool(const SpongeJob& J, const SpongeResume* R, const SpongeDual* D, uint64_t i) {
  constexpr uint64_t RATE = 8ull * LANES;
  const uint64_t state_n = R->state_n;
  uint64_t* bs = D->b_state;
  Lane a[25], b[25];
#pragma unroll
  for (int k = 0; k < 25; k++) {
    const uint64_t va = J.chain_in[(uint64_t)k * state_n + i], vb = bs[(uint64_t)k * state_n + i];
    a[k].lo = (uint32_t)va;
    a[k].hi = (uint32_t)(va >> 32);
    b[k].lo = (uint32_t)vb;
    b[k].hi = (uint32_t)(vb >> 32);
  }
  const bool open = D->open != 0;
  const uint64_t p0 = R->totals[i], a0 = J.off[i], p1 = p0 + (J.off[i + 1] - a0);
  const uint8_t* x = J.data + a0;  // stream byte p goes with x[p - p0] and o[p - p0]
  uint8_t* o = D->out ? D->out + a0 : nullptr;
  const bool release = o && D->verdict[i];
  uint8_t* cb = R->carry + i * RATE;  // stream byte p of the current block s at cb[p - s]
  const bool al = ((reinterpret_cast<uintptr_t>(x) - p0) & 7u) == 0 && (!o || ((reinterpret_cast<uintptr_t>(o) - p0) & 7u) == 0);
#pragma unroll 1
  for (uint64_t s = p0 - p0 % RATE; s < p1; s += RATE) {
    const bool full = s + RATE <= p1;
#pragma unroll
    for (int j = 0; j < LANES; j++) {
      const uint64_t l0 = s + 8ull * j, lo = l0 > p0 ? l0 : p0, hi = l0 + 8 < p1 ? l0 + 8 : p1;
      const uint64_t ks = open ? ((uint64_t)a[j].hi << 32) | a[j].lo : 0ull;
      uint64_t v = 0;  // the lane of block s: carry bytes below p0, piece bytes (plaintext in the open mode) from p0 on
      if (lo < hi) {
        if (al && hi - lo == 8) {
          const uint2 m = *reinterpret_cast<const uint2*>(x + (lo - p0));
          const uint64_t c = ((uint64_t)m.y << 32) | m.x;
          v = c ^ ks;
          if (o) {
            const uint64_t w = release ? v : c;
            *reinterpret_cast<uint2*>(o + (lo - p0)) = make_uint2((uint32_t)w, (uint32_t)(w >> 32));
          }
          if (!full) *reinterpret_cast<uint2*>(cb + 8 * j) = make_uint2((uint32_t)v, (uint32_t)(v >> 32));
        } else {
#pragma unroll 1
          for (uint64_t q = lo; q < hi; q++) {
            const uint8_t c = x[q - p0], pt = c ^ (uint8_t)(ks >> (8 * (uint32_t)(q - l0)));
            if (o) o[q - p0] = release ? pt : c;
            if (!full) cb[q - s] = pt;
            v |= (uint64_t)pt << (8 * (uint32_t)(q - l0));
          }
        }
      }
      if (full) {
#pragma unroll 1
        for (uint64_t q = l0; q < p0 && q < l0 + 8; q++) v |= (uint64_t)cb[q - s] << (8 * (uint32_t)(q - l0));
        b[j].lo ^= (uint32_t)v;
        b[j].hi ^= (uint32_t)(v >> 32);
        if (!open) {
          a[j].lo ^= (uint32_t)v;
          a[j].hi ^= (uint32_t)(v >> 32);
        }
      }
    }
    if (full) {
      keccak_f1600(a);
      keccak_f1600(b);
    }
  }
#pragma unroll
  for (int k = 0; k < 25; k++) {
    J.chain_out[(uint64_t)k * state_n + i] = ((uint64_t)a[k].hi << 32) | a[k].lo;
    bs[(uint64_t)k * state_n + i] = ((uint64_t)b[k].hi << 32) | b[k].lo;
  }
  R->totals[i] = p1;
}

// the two-state path exists at the KMAC rates of D256 / 384 / 512 only (the other instantiations keep their registers)
template <int LANES>
constexpr bool kDualLanes = LANES == 17 || LANES == 19 || LANES == 21;

template <int LANES>
__global__ void __launch_bounds__(128, CAPY_SPONGE_MINB) sponge_chain_kernel(const __grid_constant__ SpongeChain C) {
  __shared__ uint32_t ticket_s;
  if (threadIdx.x == 0) ticket_s = atomicAdd(C.sync, 1u);
  __syncthreads();
  const uint32_t ticket = ticket_s, nb = C.blocks_per_job;
  const uint32_t job = ticket >= nb ? 1u : 0u, b = job ? ticket - nb : ticket;
  const SpongeJob& J = C.j[job];
  uint32_t* done = C.sync + 1 + b;
  if (job) {
    while (*reinterpret_cast<volatile uint32_t*>(done) < 4u) __nanosleep(64);
    __threadfence();
  }
  const uint64_t r = (uint64_t)b * 128 + threadIdx.x;
  if (r < J.n) {
    if (job && C.data_dependent) sponge_item<LANES, true, true>(J, sponge_rank_item(J, r), r);
    else if (kDualLanes<LANES> && C.dual.b_state) sponge_dual_resume_ool<LANES>(J, &C.resume, &C.dual, r);  // (job 0 alone)
    else if (C.resume.carry && job) sponge_squeeze_resume_ool<LANES>(J, &C.squeeze, r);  // (only encryption streams have a job 1)
    else if (C.resume.carry) sponge_item_resume_ool<LANES>(J, &C.resume, r);
    else sponge_item<LANES, true>(J, sponge_rank_item(J, r), r);
  }
  if (!job) {
    __threadfence();  // this thread's state is visible before the warp reports
    __syncwarp();
    if ((threadIdx.x & 31u) == 0) atomicAdd(done, 1u);
  }
}

// Chain-bound ragged batch in ONE launch, three tiers by rank in the length-sorted order:
//   blocks [0, warp_blocks)                        one WARP per item   ranks [0, J.warp_items)        4 items per block
//   blocks [warp_blocks, warp_blocks + pair_blocks) two threads per item ranks [J.warp_items, J.first)  64 items per block
//   the remaining blocks                            one thread per item  ranks [J.first, J.n)          128 items per block
// Blocks are dispatched in index order, so the blocks with the longest chains are resident from the start (as a
// second kernel on another stream they were starved behind the long-lived blocks of the thread-per-item kernel and
// ran after it).  Launched with one 128-thread block per SM (shared-memory throttle): a chain advances fastest with
// its scheduler to itself.
// The three tiers are compiled as separate (out-of-line) functions: inlined into one kernel body they share one
// register allocation and instruction schedule, which slowed the thread-per-item chain from 4.6 to 5.4 us per
// permutation.
template <int LANES>
__device__ __noinline__ void sponge_item_solo_ool(const SpongeJob& J, uint64_t i) { sponge_item<LANES>(J, i); }
template <int LANES>
__device__ __noinline__ void sponge_item_pair_ool(const SpongeJob& J, uint64_t i, bool valid, uint32_t half) {
  sponge_item_pair<LANES>(J, i, valid, half);
}

// block ranges of the warp tier: class c (c + 1 chains per scheduler) owns blocks [first_block[c], first_block[c + 1])
// (the last class ends at warp_blocks) and the ranks from first_rank[c], 4 (c + 1) per block
struct SpongeTiers {
  uint32_t first_block[3];
  uint64_t first_rank[3];
  uint32_t warp_blocks, pair_blocks;
};

template <int LANES>
__global__ void __launch_bounds__(384, 1) sponge_tiered_kernel(const SpongeJob J, const SpongeTiers tiers) {
  // __launch_bounds__(.., 1): with the default bound ptxas held the kernel at 128 registers and, once the unrolled
  // warp-tier permutation was part of it, scheduled the (instruction-for-instruction identical) round loop of the
  // thread tier differently: 5.4 instead of 4.6 us per permutation at one warp per scheduler.
  // blockDim.x = 384: a warp-tier block of class c runs 4 c chains (a warp-tier chain issues ~32 instructions per
  // ~180-clock round, so up to three share a scheduler), the pair and thread tiers want a scheduler per warp and use the
  // first four warps only; warps without work exit at once.
  const uint32_t warp_blocks = tiers.warp_blocks, pair_blocks = tiers.pair_blocks;
  if (blockIdx.x >= warp_blocks) {
    if (threadIdx.x >= 128) return;
    if (blockIdx.x >= warp_blocks + pair_blocks) {
      const uint64_t r = J.first + (uint64_t)(blockIdx.x - warp_blocks - pair_blocks) * 128 + threadIdx.x;
      if (r >= J.n) return;
      sponge_item_solo_ool<LANES>(J, sponge_rank_item(J, r));
    } else {
      const uint64_t t = (uint64_t)(blockIdx.x - warp_blocks) * 128 + threadIdx.x;
      const uint64_t r = J.warp_items + (t >> 1);
      const bool valid = r < J.first;  // idle pairs of the last warp still take part in the shuffles
      sponge_item_pair_ool<LANES>(J, valid ? sponge_rank_item(J, r) : 0, valid, (uint32_t)(t & 1));
    }
  } else {
    const int c = blockIdx.x >= tiers.first_block[2] ? 2 : blockIdx.x >= tiers.first_block[1] ? 1 : 0;
    const uint32_t per_block = 4u * (c + 1), w = threadIdx.x >> 5;
    if (w >= per_block) return;
    const uint64_t r = tiers.first_rank[c] + (uint64_t)(blockIdx.x - tiers.first_block[c]) * per_block + w;
    const uint64_t end = c < 2 ? tiers.first_rank[c + 1] : J.warp_items;
    if (r >= end) return;  // whole warps leave together
    sponge_item_warp<LANES>(J, sponge_rank_item(J, r));
  }
}

}  // namespace capy
