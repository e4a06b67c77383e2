// sponge_job.h -- what a sponge job is: the parameters of the sponge kernels (sponge.cuh), and the rates of the operators
// that fill them in.  No device code: the host files that build jobs include it without the kernels.
#pragma once
#include <cstdint>

namespace capy {

struct SpongeJob {
  // constant prefix segment
  const uint8_t* prefix;
  uint32_t prefix_len;
  // state after the first skip_blocks blocks (all inside P) were absorbed; nullptr = zero state
  const uint64_t* init_state;
  uint32_t skip_blocks;
  // per-item keys (nullptr = no key block).  key_off == nullptr -> fixed key_len at key_stride
  const uint8_t* keys;
  const uint64_t* key_off;
  uint64_t key_stride;
  uint32_t key_len;
  uint32_t w;  // bytepad width (SecParam::bytepad_value, lib.rs:137-144)
  // per-item messages.  off == nullptr -> fixed msg_len at msg_stride
  const uint8_t* data;
  const uint64_t* off;
  uint64_t msg_stride;
  uint64_t msg_len;
  // trailer bytes, little-endian packed, trailer_len <= 4.  sha3_suffix: trailer is 0x86 when
  // len % 136 == 135 else 0x06 (rate 136 hard-coded for every d, quirk Q2)
  uint32_t trailer;
  uint32_t trailer_len;
  uint32_t sha3_suffix;
  // fips_pad: FIPS 202 pad10*1 (0x80 is ORed into the last byte even when already aligned);
  // only used by the SHAKE extras that have no reference counterpart
  uint32_t fips_pad;
  // q4_rate != 0: reference quirk Q4 (cshake with N = S = ""): after the 0x04 trailer the buffer
  // was run through shake(): a 06|86 suffix chosen from (len % 136) and a first pad to q4_rate
  uint32_t q4_rate;
  // rate in bytes as the reference computes it ((1600 - c) / 8; 172 for D224 cSHAKE, quirk Q7)
  uint32_t rate;
  // output: out_off == nullptr -> out_bytes per item at out_stride
  uint8_t* out;
  const uint64_t* out_off;
  uint64_t out_stride;
  uint64_t out_bytes;
  uint32_t sq_lanes;  // lanes emitted per squeeze block = (1600 - d) / 64
  // optional: out = squeeze XOR xor_in (same layout as out): keystream applied in place of a second pass
  // (c = m ^ kmac_xof(ke, "", |m|, ...), sha3/encryptable.rs:41-42, ecc/encryptable.rs:45)
  const uint8_t* xor_in;
  uint64_t n;
  // optional permutation of work: item index = order ? order[r] : r for rank r (length-sorted launch)
  const uint32_t* order;
  // tiers of a chain-bound batch (sponge_tiered_kernel): ranks [0, warp_items) one warp per item,
  // [warp_items, first) two threads per item, [first, n) one thread per item
  uint64_t warp_items;
  uint64_t first;
  // chain hand-off (sponge_chain_kernel): the chains of a uniform batch are cut in two segments that run as dependent jobs.
  //   chain_out != nullptr: absorb blocks [skip_blocks, stop_block) only, then store the 25 lanes at chain_out[k * n + rank]
  //   chain_in  != nullptr: start from the lanes another segment stored there (instead of init_state), at block skip_blocks
  uint64_t* chain_out;
  const uint64_t* chain_in;
  uint64_t stop_block;
};

// Resumable streams (capy_hasher; a job of sponge_chain_kernel with order == nullptr, so rank = item i).  Item i's state
// at chain_in[k * state_n + i] holds every whole block of its stream before the carry bytes carry[i * rate ..), whose
// count is totals[i] % rate.  With chain_out the job is an update (absorbs the whole blocks of carry | X, stores the
// state, keeps the rest as the new carry, adds |X| to totals[i]); without, the final (carry | T | pad, then squeeze).
// Kept out of SpongeJob, so that the kernels without a hand-off compile to what they were.
struct SpongeResume {
  uint8_t* carry;    // nullptr: not a resumable job
  uint64_t* totals;
  uint64_t state_n;  // stride of the lane-major states (the items of the device; a job may cover a part of them)
};

// Resumable keystreams (the keystream sponge of a capy_hasher encryption stream: job 1 of sponge_chain_kernel, beside the
// update of its tag stream in job 0).  Item i's state at chain_in[k * state_n + i] is the sponge at the start of squeeze
// block pos[i] / (8 LANES): the keystream is prefix-consistent, so piece X takes keystream bytes [pos[i], pos[i] + |X|).
// The job writes out[off[i] ..) = those bytes ^ data[off[i] ..), permutes at every block end it reaches (eagerly: a piece
// that ends on a block boundary leaves the state of the next block), stores the state at chain_out and advances pos[i].
// A position of its own, not the tag stream's total: job 0 of the same launch advances that.  Kept out of SpongeJob, like
// SpongeResume.
struct SpongeSqueeze {
  uint64_t* pos;
  uint64_t state_n;
};

// Two-state resumable streams (sign and decryption streams of capy_hasher: job 0 of sponge_chain_kernel alone, beside a
// SpongeResume).  State A at chain_in / chain_out and state B at b_state[k * state_n + i] have the same rate, 8 LANES
// bytes (the KMAC rate, which at D256 / 384 / 512 is also the squeeze width), so they share the carry and the total of
// the SpongeResume and permute at the same block ends.
//   open == 0 (dual absorb, sign pass 2): every whole block of carry | X is absorbed into A and into B.
//   open != 0 (decryption): A is a keystream at the start of squeeze block totals[i] / rate; pt = X ^ keystream, and every
//     whole block of carry | pt is absorbed into B (the tag stream); the carry holds plaintext.  With out, item i writes
//     out[off[i] ..) = pt when verdict[i] != 0, else X (the ciphertext); out may be data.  Without out nothing is written
//     but the states, the carry and the total.
// Kept out of SpongeJob, like SpongeResume.
struct SpongeDual {
  uint64_t* b_state;  // nullptr: not a two-state job
  uint32_t open;
  const uint8_t* verdict;
  uint8_t* out;
};

// Copies of resumable streams (export, import and fork of SHA3-d / KMACXOF capy_hasher batches: job 0 of
// sponge_chain_kernel alone, J.n items).  Item t reads stream src ? src[t] : t of `from` and writes stream
// dst ? dst[t] : t of `to`.  A side is either a hasher's buffers (state != nullptr: 25 lanes at state[l * state_n + j],
// the carry at carry[j * rate ..), totals[j]) or item-major records of 208 + rate bytes at rec (the 25 lanes, the total,
// the carry).  Carry bytes from total % rate on are written as zero, so a record does not depend on how the stream was
// cut into pieces; a non-zero one read from records sets *bad_tail.  Kept out of SpongeJob, like SpongeResume.
struct SpongeStreams {
  uint64_t* state;
  uint8_t* carry;
  uint64_t* totals;
  uint64_t state_n;
  uint8_t* rec;
};
struct SpongeCopy {
  const uint64_t* src;  // nullptr: identity
  const uint64_t* dst;
  SpongeStreams from, to;
  int* bad_tail;        // nullptr: not checked
  uint32_t on;          // 0: not a copy job
};

// ---- rates in bytes, as the reference computes them ------------------------------------------------------------------
// SHA3-d capacity in bits: 2d rounded up to the reference's buckets (constants.rs:38-45)
inline uint32_t sha3_capacity(int d) {
  int x = d * 2;
  return x <= 448 ? 448u : x <= 512 ? 512u : x <= 768 ? 768u : 1024u;
}
// SHA3-d: 144 / 136 / 104 / 72
inline uint32_t sha3_rate(int d) { return (1600 - sha3_capacity(d)) / 8; }
// cSHAKE and KMAC run with capacity d bits (shake_functions.rs:63, quirk Q7): 172 / 168 / 152 / 136, which is also the
// bytepad width w (SecParam::bytepad_value, lib.rs:137-144)
inline uint32_t cshake_rate(int d) { return (uint32_t)(1600 - d) / 8; }
// FIPS 202 SHAKE128 / SHAKE256: 168 / 136
inline uint32_t shake_rate(int shake_bits) { return (uint32_t)(1600 - 2 * shake_bits) / 8; }
// lanes emitted per squeeze block of a sponge of capacity c bits (Rate::from(&d), sponge.rs:27)
inline uint32_t squeeze_lanes(int c) { return (uint32_t)(1600 - c) / 64; }

}  // namespace capy
