//! `capycrypt::gpu` -- batch entry points backed by libcapycrypt_gpu (B200, sm_100a).
//!
//! SOURCE-ONLY DELIVERABLE: this image has no rustc/cargo, so this file has not been compiled.  It is the
//! binding a capyCRYPT maintainer adds as `src/gpu.rs` (+ `pub mod gpu;` in `src/lib.rs` and the `build.rs`
//! next to this file).  The `extern "C"` block binds EVERY export of `include/capy_gpu.h`; it is generated from the
//! header by `tools/gen_rust_extern.py` and `tests/test_rust_shim.py` checks names, arity and parameter types of the two
//! against each other, so the block cannot drift although this file has never been through rustc.
//!
//! The existing API stays the contract: results land in the same `Message` fields the scalar
//! traits fill (`SpongeHashable::compute_sha3_hash` -> `.digest`, `Signable::sign` -> `.sig`, `.d`).
use crate::{ecc::keypair::KeyPair, ecc::signable::Signature, Message, OperationError, SecParam};
use std::os::raw::{c_char, c_int, c_void};
use tiny_ed448_goldilocks::curve::{extended_edwards::ExtendedPoint, field::scalar::Scalar};

#[repr(C)]
pub struct CapyCtx {
    _private: [u8; 0],
}

#[repr(C)]
pub struct CapyEd448Pub {
    _private: [u8; 0],
}

#[repr(C)]
pub struct CapyHasher {
    _private: [u8; 0],
}

#[link(name = "capycrypt_gpu", kind = "static")]
extern "C" {
    fn capy_gpu_init(devices: *const c_int, n_devices: c_int, out_ctx: *mut *mut CapyCtx) -> c_int;
    fn capy_gpu_destroy(ctx: *mut CapyCtx);
    fn capy_gpu_device_count(ctx: *const CapyCtx) -> c_int;
    fn capy_gpu_scrub(ctx: *mut CapyCtx) -> c_int;
    fn capy_strerror(status: c_int) -> *const c_char;
    fn capy_last_cuda_error(ctx: *const CapyCtx) -> *const c_char;
    fn capy_version() -> c_int;
    fn capy_host_alloc(bytes: usize) -> *mut c_void;
    fn capy_host_free(p: *mut c_void);
    fn capy_copy_probe(ctx: *mut CapyCtx, dev_index: c_int, h_in: *const c_void, in_bytes: usize, h_out: *mut c_void,
        out_bytes: usize, reps: c_int, ms_per_rep: *mut f64) -> c_int;
    fn capy_launch_count(ctx: *const CapyCtx) -> u64;
    fn capy_gpu_set_plan_cache(ctx: *mut CapyCtx, enable: c_int) -> c_int;
    fn capy_plan_tiers(items_longer_than: *const u32, n_bins: u32, n: u64, max_blocks: u32, total_blocks: u64,
        sm_count: c_int, warp_items: *mut u64, pair_items: *mut u64) -> c_int;
    fn capy_plan_tiers3(items_longer_than: *const u32, n_bins: u32, n: u64, max_blocks: u32, total_blocks: u64,
        sm_count: c_int, warp_items_by_sharing: *mut u64, pair_items: *mut u64) -> c_int;
    fn capy_chain_cut(sm_count: c_int, n: u64, absorb_blocks: u64, squeeze_extra: u64,
        cut_after_blocks: *mut u64) -> c_int;
    fn capy_lpt_shares(off: *const u64, n: u64, parts: u32, unit_bytes: u32, per_item_cost: u64,
        owner: *mut u32) -> c_int;
    fn capy_sha3_batch(ctx: *mut CapyCtx, d_bits: c_int, data: *const u8, off: *const u64, n: u64, digests: *mut u8,
        flags: u32) -> c_int;
    fn capy_sha3_batch_fixed(ctx: *mut CapyCtx, d_bits: c_int, data: *const u8, msg_len: u64, stride: u64, n: u64,
        digests: *mut u8, flags: u32) -> c_int;
    fn capy_sha3_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_data: *const u8, d_off: *const u64, n: u64, d_digests: *mut u8, flags: u32) -> c_int;
    fn capy_sha3_batch_fixed_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_data: *const u8, msg_len: u64, stride: u64, n: u64, d_digests: *mut u8, flags: u32) -> c_int;
    fn capy_cshake_batch(ctx: *mut CapyCtx, d_bits: c_int, data: *const u8, off: *const u64, n: u64,
        fn_name: *const u8, fn_len: u32, custom: *const u8, custom_len: u32, out_bits: u64, out: *mut u8) -> c_int;
    fn capy_cshake_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_data: *const u8, d_off: *const u64, n: u64, fn_name: *const u8, fn_len: u32, custom: *const u8,
        custom_len: u32, out_bits: u64, d_out: *mut u8) -> c_int;
    fn capy_kmac_xof_batch(ctx: *mut CapyCtx, d_bits: c_int, keys: *const u8, key_off: *const u64, data: *const u8,
        off: *const u64, n: u64, custom: *const u8, custom_len: u32, out_bits: u64, out_off: *const u64,
        out: *mut u8) -> c_int;
    fn capy_kmac_xof_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_keys: *const u8, d_key_off: *const u64, d_data: *const u8, d_off: *const u64, n: u64, custom: *const u8,
        custom_len: u32, out_bits: u64, d_out_off: *const u64, d_out: *mut u8) -> c_int;
    fn capy_kmac_xof_batch_fixed_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_keys: *const u8, key_len: u64, key_stride: u64, d_data: *const u8, msg_len: u64, msg_stride: u64, n: u64,
        custom: *const u8, custom_len: u32, out_bits: u64, d_out: *mut u8) -> c_int;
    fn capy_fips_shake_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, shake_bits: c_int,
        d_data: *const u8, d_off: *const u64, n: u64, out_bytes: u64, d_out: *mut u8) -> c_int;
    fn capy_ed448_fixed_base_batch(ctx: *mut CapyCtx, scalars_be56: *const u8, n: u64, out_xy112: *mut u8) -> c_int;
    fn capy_ed448_fixed_base_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void,
        d_scalars_be56: *const u8, n: u64, d_out_xy112: *mut u8) -> c_int;
    fn capy_ed448_var_base_batch(ctx: *mut CapyCtx, scalars_be56: *const u8, points_xy112: *const u8, n: u64,
        out_xy112: *mut u8) -> c_int;
    fn capy_ed448_var_base_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void,
        d_scalars_be56: *const u8, d_points_xy112: *const u8, n: u64, d_out_xy112: *mut u8,
        d_bad_flag: *mut c_int) -> c_int;
    fn capy_ed448_keygen_batch(ctx: *mut CapyCtx, d_bits: c_int, pws: *const u8, pw_off: *const u64, n: u64,
        out_xy112: *mut u8) -> c_int;
    fn capy_ed448_keygen_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_pws: *const u8, d_pw_off: *const u64, n: u64, d_out_xy112: *mut u8) -> c_int;
    fn capy_ed448_sign_batch(ctx: *mut CapyCtx, d_bits: c_int, pws: *const u8, pw_off: *const u64, msgs: *const u8,
        msg_off: *const u64, n: u64, h56: *mut u8, z_be56: *mut u8) -> c_int;
    fn capy_ed448_sign_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_pws: *const u8, d_pw_off: *const u64, d_msgs: *const u8, d_msg_off: *const u64, n: u64, d_h56: *mut u8,
        d_z_be56: *mut u8) -> c_int;
    fn capy_ed448_verify_batch(ctx: *mut CapyCtx, d_bits: c_int, pub_xy112: *const u8, msgs: *const u8,
        msg_off: *const u64, h56: *const u8, z_be56: *const u8, n: u64, ok: *mut u8) -> c_int;
    fn capy_ed448_verify_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_pub_xy112: *const u8, d_msgs: *const u8, d_msg_off: *const u64, d_h56: *const u8, d_z_be56: *const u8,
        n: u64, d_ok: *mut u8, d_bad_flag: *mut c_int) -> c_int;
    fn capy_ed448_ecdh_batch(ctx: *mut CapyCtx, k_rand56: *const u8, pub_xy112: *const u8, n: u64, wx56: *mut u8,
        z_xy112: *mut u8) -> c_int;
    fn capy_sponge_encrypt_batch(ctx: *mut CapyCtx, d_bits: c_int, variant: c_int, pws: *const u8,
        pw_off: *const u64, nonces: *const u8, nonce_len: u64, msgs: *const u8, msg_off: *const u64, n: u64,
        ct: *mut u8, tag64: *mut u8) -> c_int;
    fn capy_sponge_decrypt_batch(ctx: *mut CapyCtx, d_bits: c_int, variant: c_int, pws: *const u8,
        pw_off: *const u64, nonces: *const u8, nonce_len: u64, ct: *const u8, ct_off: *const u64, tag64: *const u8,
        n: u64, out: *mut u8, ok: *mut u8) -> c_int;
    fn capy_sponge_encrypt_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        variant: c_int, d_pws: *const u8, d_pw_off: *const u64, pw_bytes: u64, d_nonces: *const u8, nonce_len: u64,
        d_msgs: *const u8, d_msg_off: *const u64, n: u64, d_ct: *mut u8, d_tag64: *mut u8) -> c_int;
    fn capy_sponge_decrypt_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        variant: c_int, d_pws: *const u8, d_pw_off: *const u64, pw_bytes: u64, d_nonces: *const u8, nonce_len: u64,
        d_ct: *const u8, d_ct_off: *const u64, d_tag64: *const u8, n: u64, d_out: *mut u8, d_ok: *mut u8) -> c_int;
    fn capy_ed448_key_encrypt_batch(ctx: *mut CapyCtx, d_bits: c_int, pub_xy112: *const u8, k_rand56: *const u8,
        msgs: *const u8, msg_off: *const u64, n: u64, ct: *mut u8, tag56: *mut u8, z_xy112: *mut u8) -> c_int;
    fn capy_ed448_key_decrypt_batch(ctx: *mut CapyCtx, d_bits: c_int, pws: *const u8, pw_off: *const u64,
        z_xy112: *const u8, ct: *const u8, ct_off: *const u64, tag56: *const u8, n: u64, out: *mut u8,
        ok: *mut u8) -> c_int;
    fn capy_ed448_key_encrypt_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_pub_xy112: *const u8, d_k_rand56: *const u8, d_msgs: *const u8, d_msg_off: *const u64, n: u64,
        d_ct: *mut u8, d_tag56: *mut u8, d_z_xy112: *mut u8, d_bad_flag: *mut c_int) -> c_int;
    fn capy_ed448_key_decrypt_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        d_pws: *const u8, d_pw_off: *const u64, d_z_xy112: *const u8, d_ct: *const u8, d_ct_off: *const u64,
        d_tag56: *const u8, n: u64, d_out: *mut u8, d_ok: *mut u8, d_bad_flag: *mut c_int) -> c_int;
    fn capy_ed448_pub_prepare(ctx: *mut CapyCtx, pub_xy112: *const u8, out_key: *mut *mut CapyEd448Pub) -> c_int;
    fn capy_ed448_pub_uses_comb(key: *const CapyEd448Pub) -> c_int;
    fn capy_ed448_pub_free(key: *mut CapyEd448Pub);
    fn capy_ed448_verify_prepared_batch(ctx: *mut CapyCtx, d_bits: c_int, key: *const CapyEd448Pub, msgs: *const u8,
        msg_off: *const u64, h56: *const u8, z_be56: *const u8, n: u64, ok: *mut u8) -> c_int;
    fn capy_ed448_verify_prepared_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void, d_bits: c_int,
        key: *const CapyEd448Pub, d_msgs: *const u8, d_msg_off: *const u64, d_h56: *const u8, d_z_be56: *const u8,
        n: u64, d_ok: *mut u8) -> c_int;
    fn capy_ed448_key_encrypt_prepared_batch(ctx: *mut CapyCtx, d_bits: c_int, key: *const CapyEd448Pub,
        k_rand56: *const u8, msgs: *const u8, msg_off: *const u64, n: u64, ct: *mut u8, tag56: *mut u8,
        z_xy112: *mut u8) -> c_int;
    fn capy_ed448_key_encrypt_prepared_batch_dev(ctx: *mut CapyCtx, dev_index: c_int, stream: *mut c_void,
        d_bits: c_int, key: *const CapyEd448Pub, d_k_rand56: *const u8, d_msgs: *const u8, d_msg_off: *const u64,
        n: u64, d_ct: *mut u8, d_tag56: *mut u8, d_z_xy112: *mut u8) -> c_int;
    fn capy_sha3_hasher_new(ctx: *mut CapyCtx, d_bits: c_int, n: u64, out: *mut *mut CapyHasher) -> c_int;
    fn capy_kmac_xof_hasher_new(ctx: *mut CapyCtx, d_bits: c_int, keys: *const u8, key_off: *const u64, n: u64,
        custom: *const u8, custom_len: u32, out: *mut *mut CapyHasher) -> c_int;
    fn capy_hasher_device_range(h: *const CapyHasher, dev_index: c_int, i0: *mut u64, i1: *mut u64) -> c_int;
    fn capy_hasher_update(ctx: *mut CapyCtx, h: *mut CapyHasher, data: *const u8, off: *const u64) -> c_int;
    fn capy_hasher_update_dev(ctx: *mut CapyCtx, h: *mut CapyHasher, dev_index: c_int, stream: *mut c_void,
        d_data: *const u8, d_off: *const u64) -> c_int;
    fn capy_hasher_final(ctx: *mut CapyCtx, h: *mut CapyHasher, out_bits: u64, out_off: *const u64,
        out: *mut u8) -> c_int;
    fn capy_hasher_final_dev(ctx: *mut CapyCtx, h: *mut CapyHasher, dev_index: c_int, stream: *mut c_void,
        out_bits: u64, d_out_off: *const u64, d_out: *mut u8) -> c_int;
    fn capy_hasher_free(h: *mut CapyHasher);
    fn capy_sponge_encrypt_stream_new(ctx: *mut CapyCtx, d_bits: c_int, variant: c_int, pws: *const u8,
        pw_off: *const u64, nonces: *const u8, nonce_len: u64, n: u64, out: *mut *mut CapyHasher) -> c_int;
    fn capy_ed448_key_encrypt_stream_new(ctx: *mut CapyCtx, d_bits: c_int, pub_xy112: *const u8,
        key: *const CapyEd448Pub, k_rand56: *const u8, n: u64, z_xy112: *mut u8, out: *mut *mut CapyHasher) -> c_int;
    fn capy_ed448_verify_stream_new(ctx: *mut CapyCtx, d_bits: c_int, pub_xy112: *const u8, key: *const CapyEd448Pub,
        h56: *const u8, z_be56: *const u8, n: u64, out: *mut *mut CapyHasher) -> c_int;
    fn capy_hasher_encrypt_update(ctx: *mut CapyCtx, h: *mut CapyHasher, data: *const u8, off: *const u64,
        ct: *mut u8) -> c_int;
    fn capy_hasher_encrypt_update_dev(ctx: *mut CapyCtx, h: *mut CapyHasher, dev_index: c_int, stream: *mut c_void,
        d_data: *const u8, d_off: *const u64, d_ct: *mut u8) -> c_int;
    fn capy_hasher_verify_final(ctx: *mut CapyCtx, h: *mut CapyHasher, ok: *mut u8) -> c_int;
    fn capy_hasher_verify_final_dev(ctx: *mut CapyCtx, h: *mut CapyHasher, dev_index: c_int, stream: *mut c_void,
        d_ok: *mut u8, d_bad_flag: *mut c_int) -> c_int;
    fn capy_ed448_sign_stream_new(ctx: *mut CapyCtx, d_bits: c_int, pws: *const u8, pw_off: *const u64, n: u64,
        out: *mut *mut CapyHasher) -> c_int;
    fn capy_sponge_decrypt_stream_new(ctx: *mut CapyCtx, d_bits: c_int, variant: c_int, pws: *const u8,
        pw_off: *const u64, nonces: *const u8, nonce_len: u64, tag64: *const u8, n: u64,
        out: *mut *mut CapyHasher) -> c_int;
    fn capy_ed448_key_decrypt_stream_new(ctx: *mut CapyCtx, d_bits: c_int, pws: *const u8, pw_off: *const u64,
        z_xy112: *const u8, tag56: *const u8, n: u64, out: *mut *mut CapyHasher) -> c_int;
    fn capy_hasher_next_pass(ctx: *mut CapyCtx, h: *mut CapyHasher, ok: *mut u8) -> c_int;
    fn capy_hasher_next_pass_dev(ctx: *mut CapyCtx, h: *mut CapyHasher, dev_index: c_int, stream: *mut c_void,
        d_ok: *mut u8, d_bad_flag: *mut c_int) -> c_int;
    fn capy_hasher_decrypt_update(ctx: *mut CapyCtx, h: *mut CapyHasher, ct: *const u8, off: *const u64,
        out: *mut u8) -> c_int;
    fn capy_hasher_decrypt_update_dev(ctx: *mut CapyCtx, h: *mut CapyHasher, dev_index: c_int, stream: *mut c_void,
        d_ct: *const u8, d_off: *const u64, d_out: *mut u8) -> c_int;
    fn capy_hasher_decrypt_final(ctx: *mut CapyCtx, h: *mut CapyHasher, ok: *mut u8) -> c_int;
    fn capy_hasher_decrypt_final_dev(ctx: *mut CapyCtx, h: *mut CapyHasher, dev_index: c_int, stream: *mut c_void,
        d_ok: *mut u8, d_bad_flag: *mut c_int) -> c_int;
    fn capy_hasher_sign_final(ctx: *mut CapyCtx, h: *mut CapyHasher, h56: *mut u8, z_be56: *mut u8,
        ok: *mut u8) -> c_int;
    fn capy_hasher_sign_final_dev(ctx: *mut CapyCtx, h: *mut CapyHasher, dev_index: c_int, stream: *mut c_void,
        d_h56: *mut u8, d_z_be56: *mut u8, d_ok: *mut u8) -> c_int;
}

const CAPY_AE_SHA3: c_int = 0;

/// affine (x || y, 2 x 56 little-endian bytes) of an `ExtendedPoint` -- the point format of the C ABI
fn point_to_xy(p: &ExtendedPoint) -> [u8; 112] {
    let a = p.to_affine();
    let mut o = [0u8; 112];
    o[..56].copy_from_slice(&a.x.to_bytes());
    o[56..].copy_from_slice(&a.y.to_bytes());
    o
}

/// One engine context (one or more GPUs).  Calls are blocking and serialised per context.
pub struct Gpu {
    ctx: *mut CapyCtx,
}
unsafe impl Send for Gpu {}

fn pack<'a, I: Iterator<Item = &'a [u8]>>(items: I) -> (Vec<u8>, Vec<u64>) {
    let mut data = Vec::new();
    let mut off = vec![0u64];
    for it in items {
        data.extend_from_slice(it);
        off.push(data.len() as u64);
    }
    if data.is_empty() {
        data.push(0);
    }
    (data, off)
}

fn status(rc: c_int) -> Result<(), OperationError> {
    match rc {
        0 => Ok(()),
        -1 => Err(OperationError::UnsupportedSecurityParameter),
        _ => Err(OperationError::OperationResultNotSet),
    }
}

impl Gpu {
    /// `devices = &[]` uses the current CUDA device.
    pub fn new(devices: &[i32]) -> Result<Gpu, OperationError> {
        let mut ctx = std::ptr::null_mut();
        let rc = unsafe {
            capy_gpu_init(if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() },
                          devices.len() as c_int, &mut ctx)
        };
        status(rc)?;
        Ok(Gpu { ctx })
    }

    /// Batched `SpongeHashable::compute_sha3_hash`: fills `Message.digest`.  `Message.msg` is also left
    /// suffixed + padded exactly as `shake()` leaves it (strict drop-in, reference quirk Q5).
    pub fn compute_sha3_hash(&self, msgs: &mut [Message], d: SecParam) -> Result<(), OperationError> {
        let (data, off) = pack(msgs.iter().map(|m| m.msg.as_slice()));
        let ob = d as usize / 8;
        let mut out = vec![0u8; msgs.len() * ob];
        status(unsafe {
            capy_sha3_batch(self.ctx, d as c_int, data.as_ptr(), off.as_ptr(), msgs.len() as u64, out.as_mut_ptr(), 0)
        })?;
        for (m, dg) in msgs.iter_mut().zip(out.chunks_exact(ob)) {
            m.digest = dg.to_vec();
            // replicate the in-place append of shake(): suffix chosen with rate 136, pad only if unaligned
            let suffix = if m.msg.len() % 136 == 135 { 0x86 } else { 0x06 };
            m.msg.push(suffix);
            let r = (1600 - 2 * (d as usize).max(224)) / 8; // capacity 2d bucketed: 144/136/104/72
            if m.msg.len() % r != 0 {
                let q = r - m.msg.len() % r;
                m.msg.extend(std::iter::repeat(0).take(q - 1));
                m.msg.push(0x80);
            }
        }
        Ok(())
    }

    /// Batched `SpongeHashable::compute_tagged_hash`.
    pub fn compute_tagged_hash(&self, msgs: &mut [Message], pws: &[&[u8]], s: &str, d: SecParam) -> Result<(), OperationError> {
        let (kd, ko) = pack(pws.iter().copied());
        let (xd, xo) = pack(msgs.iter().map(|m| m.msg.as_slice()));
        let ob = d as usize / 8;
        let mut out = vec![0u8; msgs.len() * ob];
        status(unsafe {
            capy_kmac_xof_batch(self.ctx, d as c_int, kd.as_ptr(), ko.as_ptr(), xd.as_ptr(), xo.as_ptr(),
                                msgs.len() as u64, s.as_ptr(), s.len() as u32, d as u64, std::ptr::null(), out.as_mut_ptr())
        })?;
        for (m, dg) in msgs.iter_mut().zip(out.chunks_exact(ob)) {
            m.digest = dg.to_vec();
        }
        Ok(())
    }

    /// Batched public-key derivation of `KeyPair::new`; returns affine (x, y) as 2 x 56 little-endian bytes.
    /// Build `ExtendedPoint`s with `AffinePoint { x, y }.to_extended()` (field decoding is crate-specific).
    pub fn keygen_affine(&self, pws: &[&[u8]], d: SecParam) -> Result<Vec<[u8; 112]>, OperationError> {
        let (pd, po) = pack(pws.iter().copied());
        let mut out = vec![0u8; pws.len() * 112];
        status(unsafe { capy_ed448_keygen_batch(self.ctx, d as c_int, pd.as_ptr(), po.as_ptr(), pws.len() as u64, out.as_mut_ptr()) })?;
        Ok(out.chunks_exact(112).map(|c| c.try_into().unwrap()).collect())
    }

    /// Batched `Signable::sign`: message i is signed under `keys[i]`.
    pub fn sign(&self, msgs: &mut [Message], keys: &[&KeyPair], d: SecParam) -> Result<(), OperationError> {
        let (pd, po) = pack(keys.iter().map(|k| k.priv_key.as_slice()));
        let (md, mo) = pack(msgs.iter().map(|m| m.msg.as_slice()));
        let n = msgs.len();
        let (mut h, mut z) = (vec![0u8; n * 56], vec![0u8; n * 56]);
        status(unsafe {
            capy_ed448_sign_batch(self.ctx, d as c_int, pd.as_ptr(), po.as_ptr(), md.as_ptr(), mo.as_ptr(), n as u64,
                                  h.as_mut_ptr(), z.as_mut_ptr())
        })?;
        for (i, m) in msgs.iter_mut().enumerate() {
            let z_scalar = Scalar { val: crypto_bigint::U448::from_be_slice(&z[56 * i..56 * i + 56]) };
            m.sig = Some(Signature { h: h[56 * i..56 * i + 56].to_vec(), z: z_scalar });
            m.d = Some(d);
        }
        Ok(())
    }

    /// Batched `Signable::verify`; `pub_keys[i]` verifies `msgs[i]`.  Same errors as src/ecc/signable.rs:72-86.
    pub fn verify(&self, msgs: &[Message], pub_keys: &[ExtendedPoint]) -> Vec<Result<(), OperationError>> {
        let mut res: Vec<Result<(), OperationError>> = msgs.iter().map(|_| Ok(())).collect();
        for d in [SecParam::D224, SecParam::D256, SecParam::D384, SecParam::D512] {
            let mut idx = Vec::new();
            for (i, m) in msgs.iter().enumerate() {
                if m.sig.is_none() {
                    res[i] = Err(OperationError::SignatureNotSet);
                } else if m.d.is_none() {
                    res[i] = Err(OperationError::SecurityParameterNotSet);
                } else if m.d == Some(d) {
                    idx.push(i);
                }
            }
            if idx.is_empty() {
                continue;
            }
            let (mut pk, mut h, mut z) = (Vec::new(), Vec::new(), Vec::new());
            // a signature whose h is not 56 bytes fails on its own and stays out of the fixed-stride batch (one short
            // field would shift every later item and make the C side read past the Vec)
            idx.retain(|&i| {
                let good = msgs[i].sig.as_ref().unwrap().h.len() == 56;
                if !good {
                    res[i] = Err(OperationError::SignatureVerificationFailure);
                }
                good
            });
            if idx.is_empty() {
                continue;
            }
            for &i in &idx {
                let sig = msgs[i].sig.as_ref().unwrap();
                pk.extend_from_slice(&point_to_xy(&pub_keys[i]));
                h.extend_from_slice(&sig.h);
                z.extend_from_slice(&sig.z.val.to_be_bytes());
            }
            debug_assert!(pk.len() == 112 * idx.len() && h.len() == 56 * idx.len() && z.len() == 56 * idx.len());
            let (md, mo) = pack(idx.iter().map(|&i| msgs[i].msg.as_slice()));
            let mut ok = vec![0u8; idx.len()];
            let rc = unsafe {
                capy_ed448_verify_batch(self.ctx, d as c_int, pk.as_ptr(), md.as_ptr(), mo.as_ptr(), h.as_ptr(), z.as_ptr(),
                                        idx.len() as u64, ok.as_mut_ptr())
            };
            for (k, &i) in idx.iter().enumerate() {
                if (rc != 0 && rc != -4) || ok[k] == 0 {
                    res[i] = Err(OperationError::SignatureVerificationFailure);
                }
            }
        }
        res
    }

    /// Batched `SpongeEncryptable::sha3_encrypt` (src/sha3/encryptable.rs:29-45).  The 512 random nonce bytes per
    /// message are drawn here with the reference's own `get_random_bytes` (the C ABI has no RNG).
    pub fn sha3_encrypt(&self, msgs: &mut [Message], pws: &[&[u8]], d: SecParam) -> Result<(), OperationError> {
        use crate::sha3::aux_functions::byte_utils::get_random_bytes;
        let n = msgs.len();
        let nonces: Vec<Vec<u8>> = (0..n).map(|_| get_random_bytes(512)).collect();
        let z: Vec<u8> = nonces.iter().flatten().copied().collect();
        let (pd, po) = pack(pws.iter().copied());
        let (md, mo) = pack(msgs.iter().map(|m| m.msg.as_slice()));
        let (mut ct, mut tag) = (vec![0u8; md.len()], vec![0u8; n * 64]);
        status(unsafe {
            capy_sponge_encrypt_batch(self.ctx, d as c_int, CAPY_AE_SHA3, pd.as_ptr(), po.as_ptr(), z.as_ptr(), 512,
                                      md.as_ptr(), mo.as_ptr(), n as u64, ct.as_mut_ptr(), tag.as_mut_ptr())
        })?;
        for (i, (m, nonce)) in msgs.iter_mut().zip(nonces).enumerate() {
            m.msg = Box::new(ct[mo[i] as usize..mo[i + 1] as usize].to_vec());
            m.digest = tag[64 * i..64 * i + 64].to_vec();
            m.sym_nonce = Some(nonce);
            m.d = Some(d);
        }
        Ok(())
    }

    /// Batched `SpongeEncryptable::sha3_decrypt` (:58-83): on `SHA3DecryptionFailure` the message keeps its ciphertext.
    pub fn sha3_decrypt(&self, msgs: &mut [Message], pws: &[&[u8]]) -> Vec<Result<(), OperationError>> {
        let mut res: Vec<Result<(), OperationError>> = msgs.iter().map(|_| Ok(())).collect();
        // one C call per (d, nonce length): the C side reads n * nonce_len bytes, so every nonce of a call must have
        // exactly that length (a deserialized Message may carry any length; the reference would simply derive other keys)
        let mut groups: std::collections::BTreeMap<(usize, usize), Vec<usize>> = std::collections::BTreeMap::new();
        for (i, m) in msgs.iter().enumerate() {
            if m.d.is_none() {
                res[i] = Err(OperationError::SecurityParameterNotSet);
            } else if m.sym_nonce.is_none() {
                res[i] = Err(OperationError::SymNonceNotSet);
            } else {
                groups.entry((m.d.unwrap() as usize, m.sym_nonce.as_ref().unwrap().len())).or_default().push(i);
            }
        }
        for ((d_bits, nonce_len), idx) in groups {
            let d = SecParam::try_from(d_bits).unwrap();
            let (pd, po) = pack(idx.iter().map(|&i| pws[i]));
            let (cd, co) = pack(idx.iter().map(|&i| msgs[i].msg.as_slice()));
            let z: Vec<u8> = idx.iter().flat_map(|&i| msgs[i].sym_nonce.as_ref().unwrap().iter().copied()).collect();
            debug_assert!(z.len() == nonce_len * idx.len());
            let mut tags = vec![0u8; idx.len() * 64];
            for (k, &i) in idx.iter().enumerate() {
                let t = &msgs[i].digest;
                tags[64 * k..64 * k + t.len().min(64)].copy_from_slice(&t[..t.len().min(64)]);
            }
            let (mut out, mut ok) = (vec![0u8; cd.len()], vec![0u8; idx.len()]);
            let rc = unsafe {
                capy_sponge_decrypt_batch(self.ctx, d as c_int, CAPY_AE_SHA3, pd.as_ptr(), po.as_ptr(), z.as_ptr(), nonce_len as u64,
                                          cd.as_ptr(), co.as_ptr(), tags.as_ptr(), idx.len() as u64, out.as_mut_ptr(),
                                          ok.as_mut_ptr())
            };
            for (k, &i) in idx.iter().enumerate() {
                if rc == 0 && ok[k] == 1 && msgs[i].digest.len() == 64 {
                    msgs[i].msg = Box::new(out[co[k] as usize..co[k + 1] as usize].to_vec());
                } else {
                    res[i] = Err(OperationError::SHA3DecryptionFailure);
                }
            }
        }
        res
    }

    /// Batched `KeyEncryptable::key_encrypt` (src/ecc/encryptable.rs:34-50); `pub_keys[i]` encrypts `msgs[i]`.
    pub fn key_encrypt(&self, msgs: &mut [Message], pub_keys: &[ExtendedPoint], d: SecParam) -> Result<(), OperationError> {
        use crate::sha3::aux_functions::byte_utils::get_random_bytes;
        use tiny_ed448_goldilocks::curve::affine::AffinePoint;
        let n = msgs.len();
        let k_rand: Vec<u8> = (0..n).flat_map(|_| get_random_bytes(56)).collect();
        let pk: Vec<u8> = pub_keys.iter().flat_map(|p| point_to_xy(p)).collect();
        let (md, mo) = pack(msgs.iter().map(|m| m.msg.as_slice()));
        let (mut ct, mut tag, mut z) = (vec![0u8; md.len()], vec![0u8; n * 56], vec![0u8; n * 112]);
        status(unsafe {
            capy_ed448_key_encrypt_batch(self.ctx, d as c_int, pk.as_ptr(), k_rand.as_ptr(), md.as_ptr(), mo.as_ptr(),
                                         n as u64, ct.as_mut_ptr(), tag.as_mut_ptr(), z.as_mut_ptr())
        })?;
        for (i, m) in msgs.iter_mut().enumerate() {
            m.msg = Box::new(ct[mo[i] as usize..mo[i + 1] as usize].to_vec());
            m.digest = tag[56 * i..56 * i + 56].to_vec();
            // field decoding is crate-specific: FieldElement::from_bytes on the two 56-byte halves
            m.asym_nonce = Some(AffinePoint::from_xy_bytes(&z[112 * i..112 * i + 112]).to_extended());
            m.d = Some(d);
        }
        Ok(())
    }

    /// Batched `KeyEncryptable::key_decrypt` (:72-94): on `KeyDecryptionError` the message keeps its ciphertext.
    pub fn key_decrypt(&self, msgs: &mut [Message], pws: &[&[u8]]) -> Vec<Result<(), OperationError>> {
        let mut res: Vec<Result<(), OperationError>> = msgs.iter().map(|_| Ok(())).collect();
        for d in [SecParam::D224, SecParam::D256, SecParam::D384, SecParam::D512] {
            let mut idx = Vec::new();
            for (i, m) in msgs.iter().enumerate() {
                if m.asym_nonce.is_none() {
                    res[i] = Err(OperationError::SymNonceNotSet); // sic: ecc/encryptable.rs:73
                } else if m.d.is_none() {
                    res[i] = Err(OperationError::SecurityParameterNotSet);
                } else if m.d == Some(d) {
                    idx.push(i);
                }
            }
            if idx.is_empty() {
                continue;
            }
            let (pd, po) = pack(idx.iter().map(|&i| pws[i]));
            let (cd, co) = pack(idx.iter().map(|&i| msgs[i].msg.as_slice()));
            let z: Vec<u8> = idx.iter().flat_map(|&i| point_to_xy(msgs[i].asym_nonce.as_ref().unwrap())).collect();
            let mut tags = vec![0u8; idx.len() * 56];
            for (k, &i) in idx.iter().enumerate() {
                let t = &msgs[i].digest;
                tags[56 * k..56 * k + t.len().min(56)].copy_from_slice(&t[..t.len().min(56)]);
            }
            let (mut out, mut ok) = (vec![0u8; cd.len()], vec![0u8; idx.len()]);
            let rc = unsafe {
                capy_ed448_key_decrypt_batch(self.ctx, d as c_int, pd.as_ptr(), po.as_ptr(), z.as_ptr(), cd.as_ptr(),
                                             co.as_ptr(), tags.as_ptr(), idx.len() as u64, out.as_mut_ptr(), ok.as_mut_ptr())
            };
            for (k, &i) in idx.iter().enumerate() {
                if (rc == 0 || rc == -4) && ok[k] == 1 && msgs[i].digest.len() == 56 {
                    msgs[i].msg = Box::new(out[co[k] as usize..co[k + 1] as usize].to_vec());
                } else {
                    res[i] = Err(OperationError::KeyDecryptionError);
                }
            }
        }
        res
    }
}

/// A public key prepared on every device of one `Gpu` (`Gpu::prepare_public_key`): the comb table of V that
/// `Gpu::verify_prepared` and `Gpu::key_encrypt_prepared` use instead of the variable-base ladder.  Reuse it across
/// calls; drop it before the `Gpu` that prepared it.
pub struct PreparedKey {
    key: *mut CapyEd448Pub,
}
unsafe impl Send for PreparedKey {}

impl PreparedKey {
    /// false when V has a torsion component: the prepared calls then run the generic pipelines (same results)
    pub fn uses_comb(&self) -> bool {
        unsafe { capy_ed448_pub_uses_comb(self.key) == 1 }
    }
}

impl Drop for PreparedKey {
    fn drop(&mut self) {
        unsafe { capy_ed448_pub_free(self.key) }
    }
}

impl Gpu {
    /// Prepares V for many `verify_prepared` / `key_encrypt_prepared` calls (blocking, a few ms per device).
    pub fn prepare_public_key(&self, pub_key: &ExtendedPoint) -> Result<PreparedKey, OperationError> {
        let xy = point_to_xy(pub_key);
        let mut key = std::ptr::null_mut();
        status(unsafe { capy_ed448_pub_prepare(self.ctx, xy.as_ptr(), &mut key) })?;
        Ok(PreparedKey { key })
    }

    /// Batched `Signable::verify` of every message against one signer; same errors as `verify`.
    pub fn verify_prepared(&self, msgs: &[Message], key: &PreparedKey) -> Vec<Result<(), OperationError>> {
        let mut res: Vec<Result<(), OperationError>> = msgs.iter().map(|_| Ok(())).collect();
        for d in [SecParam::D224, SecParam::D256, SecParam::D384, SecParam::D512] {
            let mut idx = Vec::new();
            for (i, m) in msgs.iter().enumerate() {
                if m.sig.is_none() {
                    res[i] = Err(OperationError::SignatureNotSet);
                } else if m.d.is_none() {
                    res[i] = Err(OperationError::SecurityParameterNotSet);
                } else if m.d == Some(d) {
                    if m.sig.as_ref().unwrap().h.len() == 56 {
                        idx.push(i);
                    } else {
                        res[i] = Err(OperationError::SignatureVerificationFailure);
                    }
                }
            }
            if idx.is_empty() {
                continue;
            }
            let (mut h, mut z) = (Vec::new(), Vec::new());
            for &i in &idx {
                let sig = msgs[i].sig.as_ref().unwrap();
                h.extend_from_slice(&sig.h);
                z.extend_from_slice(&sig.z.val.to_be_bytes());
            }
            let (md, mo) = pack(idx.iter().map(|&i| msgs[i].msg.as_slice()));
            let mut ok = vec![0u8; idx.len()];
            let rc = unsafe {
                capy_ed448_verify_prepared_batch(self.ctx, d as c_int, key.key, md.as_ptr(), mo.as_ptr(), h.as_ptr(),
                                                 z.as_ptr(), idx.len() as u64, ok.as_mut_ptr())
            };
            for (k, &i) in idx.iter().enumerate() {
                if rc != 0 || ok[k] == 0 {
                    res[i] = Err(OperationError::SignatureVerificationFailure);
                }
            }
        }
        res
    }

    /// Batched `KeyEncryptable::key_encrypt` of every message to one recipient.
    pub fn key_encrypt_prepared(&self, msgs: &mut [Message], key: &PreparedKey, d: SecParam) -> Result<(), OperationError> {
        use crate::sha3::aux_functions::byte_utils::get_random_bytes;
        use tiny_ed448_goldilocks::curve::affine::AffinePoint;
        let n = msgs.len();
        let k_rand: Vec<u8> = (0..n).flat_map(|_| get_random_bytes(56)).collect();
        let (md, mo) = pack(msgs.iter().map(|m| m.msg.as_slice()));
        let (mut ct, mut tag, mut z) = (vec![0u8; md.len()], vec![0u8; n * 56], vec![0u8; n * 112]);
        status(unsafe {
            capy_ed448_key_encrypt_prepared_batch(self.ctx, d as c_int, key.key, k_rand.as_ptr(), md.as_ptr(),
                                                  mo.as_ptr(), n as u64, ct.as_mut_ptr(), tag.as_mut_ptr(), z.as_mut_ptr())
        })?;
        for (i, m) in msgs.iter_mut().enumerate() {
            m.msg = Box::new(ct[mo[i] as usize..mo[i + 1] as usize].to_vec());
            m.digest = tag[56 * i..56 * i + 56].to_vec();
            m.asym_nonce = Some(AffinePoint::from_xy_bytes(&z[112 * i..112 * i + 112]).to_extended());
            m.d = Some(d);
        }
        Ok(())
    }
}

/// A batch of resumable SHA3-d or KMACXOF streams (`Gpu::sha3_hasher`, `Gpu::kmac_xof_hasher`): `update` appends one
/// piece per stream, `finish` returns what `compute_sha3_hash` / `kmac_xof` give for the concatenated pieces.  Drop it
/// before the `Gpu` that created it.
pub struct Hasher {
    ctx: *mut CapyCtx,
    h: *mut CapyHasher,
    n: usize,
}
unsafe impl Send for Hasher {}

impl Hasher {
    /// `pieces[i]` is appended to stream i.
    pub fn update(&mut self, pieces: &[&[u8]]) -> Result<(), OperationError> {
        if pieces.len() != self.n {
            return Err(OperationError::OperationResultNotSet);
        }
        let (data, off) = pack(pieces.iter().copied());
        status(unsafe { capy_hasher_update(self.ctx, self.h, data.as_ptr(), off.as_ptr()) })
    }

    /// SHA3-d: the digests (`l_bits` = d).  KMACXOF: `l_bits` output bits per stream.  The hasher is finished after it.
    pub fn finish(&mut self, l_bits: u64) -> Result<Vec<Vec<u8>>, OperationError> {
        let ob = (l_bits / 8) as usize;
        let mut out = vec![0u8; self.n * ob + 1];
        status(unsafe { capy_hasher_final(self.ctx, self.h, l_bits, std::ptr::null(), out.as_mut_ptr()) })?;
        Ok((0..self.n).map(|i| out[i * ob..(i + 1) * ob].to_vec()).collect())
    }
}

impl Drop for Hasher {
    fn drop(&mut self) {
        unsafe { capy_hasher_free(self.h) }
    }
}

impl Gpu {
    /// n `compute_sha3_hash` streams fed in pieces (blocking).
    pub fn sha3_hasher(&self, n: usize, d: SecParam) -> Result<Hasher, OperationError> {
        let mut h = std::ptr::null_mut();
        status(unsafe { capy_sha3_hasher_new(self.ctx, d as c_int, n as u64, &mut h) })?;
        Ok(Hasher { ctx: self.ctx, h, n })
    }

    /// One `kmac_xof` stream per key with customisation string `s` (blocking); `compute_tagged_hash` is
    /// `finish(d as u64)`.  D224 is refused (capy_gpu.h: quirk Q7).
    pub fn kmac_xof_hasher(&self, keys: &[&[u8]], s: &str, d: SecParam) -> Result<Hasher, OperationError> {
        let (kd, ko) = pack(keys.iter().copied());
        let mut h = std::ptr::null_mut();
        status(unsafe {
            capy_kmac_xof_hasher_new(self.ctx, d as c_int, kd.as_ptr(), ko.as_ptr(), keys.len() as u64, s.as_ptr(),
                                     s.len() as u32, &mut h)
        })?;
        Ok(Hasher { ctx: self.ctx, h, n: keys.len() })
    }
}

/// Encryption streams (`Gpu::sha3_encrypt_stream`, `Gpu::key_encrypt_stream_prepared`): `update` returns the ciphertext of
/// one piece per message, `finish` the tags; together they are the `.msg` and `.digest` of the one-shot call on the
/// concatenated plaintext.  `nonces` holds each message's `sym_nonce` (512 bytes) or `asym_nonce` (Z, affine x || y).
/// Drop it before the `Gpu` that created it.
pub struct EncryptStream {
    ctx: *mut CapyCtx,
    h: *mut CapyHasher,
    n: usize,
    tag_bytes: usize,
    pub nonces: Vec<Vec<u8>>,
}
unsafe impl Send for EncryptStream {}

impl EncryptStream {
    pub fn update(&mut self, pieces: &[&[u8]]) -> Result<Vec<Vec<u8>>, OperationError> {
        if pieces.len() != self.n {
            return Err(OperationError::OperationResultNotSet);
        }
        let (data, off) = pack(pieces.iter().copied());
        let mut ct = vec![0u8; data.len()];
        status(unsafe { capy_hasher_encrypt_update(self.ctx, self.h, data.as_ptr(), off.as_ptr(), ct.as_mut_ptr()) })?;
        Ok((0..self.n).map(|i| ct[off[i] as usize..off[i + 1] as usize].to_vec()).collect())
    }

    /// The tags (64 bytes for sha3_encrypt, 56 for key_encrypt).  The streams are finished after it.
    pub fn finish(&mut self) -> Result<Vec<Vec<u8>>, OperationError> {
        let tb = self.tag_bytes;
        let mut out = vec![0u8; self.n * tb + 1];
        status(unsafe { capy_hasher_final(self.ctx, self.h, 8 * tb as u64, std::ptr::null(), out.as_mut_ptr()) })?;
        Ok((0..self.n).map(|i| out[i * tb..(i + 1) * tb].to_vec()).collect())
    }
}

impl Drop for EncryptStream {
    fn drop(&mut self) {
        unsafe { capy_hasher_free(self.h) }
    }
}

/// Verification streams (`Gpu::verify_stream_prepared`): `update` appends one piece per message, `finish` gives what
/// `verify_prepared` gives for the concatenated pieces.  Drop it before the `Gpu` that created it.
pub struct VerifyStream {
    ctx: *mut CapyCtx,
    h: *mut CapyHasher,
    n: usize,
}
unsafe impl Send for VerifyStream {}

impl VerifyStream {
    pub fn update(&mut self, pieces: &[&[u8]]) -> Result<(), OperationError> {
        if pieces.len() != self.n {
            return Err(OperationError::OperationResultNotSet);
        }
        let (data, off) = pack(pieces.iter().copied());
        status(unsafe { capy_hasher_update(self.ctx, self.h, data.as_ptr(), off.as_ptr()) })
    }

    pub fn finish(&mut self) -> Vec<Result<(), OperationError>> {
        let mut ok = vec![0u8; self.n + 1];
        let rc = unsafe { capy_hasher_verify_final(self.ctx, self.h, ok.as_mut_ptr()) };
        (0..self.n)
            .map(|i| if rc != 0 || ok[i] == 0 { Err(OperationError::SignatureVerificationFailure) } else { Ok(()) })
            .collect()
    }
}

impl Drop for VerifyStream {
    fn drop(&mut self) {
        unsafe { capy_hasher_free(self.h) }
    }
}

/// n signatures whose messages are fed twice in pieces (`Gpu::sign_stream`): `update` in pass 1, `next_pass`, `update`
/// with the same bytes in pass 2, then `finish`.  An item whose two passes differ gets `OperationResultNotSet` and no
/// signature.
pub struct SignStream {
    ctx: *mut CapyCtx,
    h: *mut CapyHasher,
    n: usize,
}
unsafe impl Send for SignStream {}

impl SignStream {
    pub fn update(&mut self, pieces: &[&[u8]]) -> Result<(), OperationError> {
        if pieces.len() != self.n {
            return Err(OperationError::OperationResultNotSet);
        }
        let (data, off) = pack(pieces.iter().copied());
        status(unsafe { capy_hasher_update(self.ctx, self.h, data.as_ptr(), off.as_ptr()) })
    }

    pub fn next_pass(&mut self) -> Result<(), OperationError> {
        status(unsafe { capy_hasher_next_pass(self.ctx, self.h, std::ptr::null_mut()) })
    }

    pub fn finish(&mut self) -> Vec<Result<Signature, OperationError>> {
        let (mut h, mut z, mut ok) = (vec![0u8; self.n * 56 + 1], vec![0u8; self.n * 56 + 1], vec![0u8; self.n + 1]);
        let rc = unsafe { capy_hasher_sign_final(self.ctx, self.h, h.as_mut_ptr(), z.as_mut_ptr(), ok.as_mut_ptr()) };
        (0..self.n)
            .map(|i| {
                if rc != 0 || ok[i] == 0 {
                    return Err(OperationError::OperationResultNotSet);
                }
                let z_scalar = Scalar { val: crypto_bigint::U448::from_be_slice(&z[56 * i..56 * i + 56]) };
                Ok(Signature { h: h[56 * i..56 * i + 56].to_vec(), z: z_scalar })
            })
            .collect()
    }
}

impl Drop for SignStream {
    fn drop(&mut self) {
        unsafe { capy_hasher_free(self.h) }
    }
}

/// n decryptions whose ciphertexts are fed twice in pieces (`Gpu::sha3_decrypt_stream` / `key_decrypt_stream`):
/// `update` in pass 1, `next_pass` (the verdicts), `decrypt` with the same bytes in pass 2 (plaintext where the verdict
/// was good, the ciphertext elsewhere), then `finish`.
pub struct DecryptStream {
    ctx: *mut CapyCtx,
    h: *mut CapyHasher,
    n: usize,
    key: bool, // key_decrypt (KeyDecryptionError) rather than sha3_decrypt (SHA3DecryptionFailure)
}
unsafe impl Send for DecryptStream {}

impl DecryptStream {
    pub fn update(&mut self, pieces: &[&[u8]]) -> Result<(), OperationError> {
        if pieces.len() != self.n {
            return Err(OperationError::OperationResultNotSet);
        }
        let (data, off) = pack(pieces.iter().copied());
        status(unsafe { capy_hasher_update(self.ctx, self.h, data.as_ptr(), off.as_ptr()) })
    }

    fn verdicts(&self, rc: c_int, ok: &[u8]) -> Vec<Result<(), OperationError>> {
        let err = || if self.key { OperationError::KeyDecryptionError } else { OperationError::SHA3DecryptionFailure };
        (0..self.n).map(|i| if rc != 0 || ok[i] == 0 { Err(err()) } else { Ok(()) }).collect()
    }

    pub fn next_pass(&mut self) -> Vec<Result<(), OperationError>> {
        let mut ok = vec![0u8; self.n + 1];
        let rc = unsafe { capy_hasher_next_pass(self.ctx, self.h, ok.as_mut_ptr()) };
        self.verdicts(rc, &ok)
    }

    pub fn decrypt(&mut self, pieces: &[&[u8]]) -> Result<Vec<Vec<u8>>, OperationError> {
        if pieces.len() != self.n {
            return Err(OperationError::OperationResultNotSet);
        }
        let (data, off) = pack(pieces.iter().copied());
        let mut out = vec![0u8; data.len()];
        status(unsafe { capy_hasher_decrypt_update(self.ctx, self.h, data.as_ptr(), off.as_ptr(), out.as_mut_ptr()) })?;
        Ok((0..self.n).map(|i| out[off[i] as usize..off[i + 1] as usize].to_vec()).collect())
    }

    pub fn finish(&mut self) -> Vec<Result<(), OperationError>> {
        let mut ok = vec![0u8; self.n + 1];
        let rc = unsafe { capy_hasher_decrypt_final(self.ctx, self.h, ok.as_mut_ptr()) };
        self.verdicts(rc, &ok)
    }
}

impl Drop for DecryptStream {
    fn drop(&mut self) {
        unsafe { capy_hasher_free(self.h) }
    }
}

impl Gpu {
    /// One `sha3_encrypt` per password whose plaintext arrives in pieces (blocking); the 512 nonce bytes per message are
    /// drawn with the reference's `get_random_bytes`.  D224 is refused (capy_gpu.h: quirk Q7).
    pub fn sha3_encrypt_stream(&self, pws: &[&[u8]], d: SecParam) -> Result<EncryptStream, OperationError> {
        use crate::sha3::aux_functions::byte_utils::get_random_bytes;
        let n = pws.len();
        let nonces: Vec<Vec<u8>> = (0..n).map(|_| get_random_bytes(512)).collect();
        let z: Vec<u8> = nonces.iter().flatten().copied().collect();
        let (pd, po) = pack(pws.iter().copied());
        let mut h = std::ptr::null_mut();
        status(unsafe {
            capy_sponge_encrypt_stream_new(self.ctx, d as c_int, CAPY_AE_SHA3, pd.as_ptr(), po.as_ptr(), z.as_ptr(), 512,
                                           n as u64, &mut h)
        })?;
        Ok(EncryptStream { ctx: self.ctx, h, n, tag_bytes: 64, nonces })
    }

    /// n `key_encrypt`s to one prepared key whose plaintexts arrive in pieces (blocking); `nonces` holds each Z.
    pub fn key_encrypt_stream_prepared(&self, n: usize, key: &PreparedKey, d: SecParam)
                                       -> Result<EncryptStream, OperationError> {
        use crate::sha3::aux_functions::byte_utils::get_random_bytes;
        let k_rand: Vec<u8> = (0..n).flat_map(|_| get_random_bytes(56)).collect();
        let mut z = vec![0u8; n * 112 + 1];
        let mut h = std::ptr::null_mut();
        status(unsafe {
            capy_ed448_key_encrypt_stream_new(self.ctx, d as c_int, std::ptr::null(), key.key, k_rand.as_ptr(), n as u64,
                                              z.as_mut_ptr(), &mut h)
        })?;
        let nonces = (0..n).map(|i| z[112 * i..112 * (i + 1)].to_vec()).collect();
        Ok(EncryptStream { ctx: self.ctx, h, n, tag_bytes: 56, nonces })
    }

    /// `verify_prepared` of signatures whose messages arrive in pieces (blocking).
    pub fn verify_stream_prepared(&self, sigs: &[Signature], key: &PreparedKey, d: SecParam)
                                  -> Result<VerifyStream, OperationError> {
        let (mut h, mut z) = (Vec::new(), Vec::new());
        for sig in sigs {
            if sig.h.len() != 56 {
                return Err(OperationError::SignatureVerificationFailure);
            }
            h.extend_from_slice(&sig.h);
            z.extend_from_slice(&sig.z.val.to_be_bytes());
        }
        h.push(0);
        z.push(0);
        let mut hs = std::ptr::null_mut();
        status(unsafe {
            capy_ed448_verify_stream_new(self.ctx, d as c_int, std::ptr::null(), key.key, h.as_ptr(), z.as_ptr(),
                                         sigs.len() as u64, &mut hs)
        })?;
        Ok(VerifyStream { ctx: self.ctx, h: hs, n: sigs.len() })
    }
}

impl Drop for Gpu {
    fn drop(&mut self) {
        unsafe { capy_gpu_destroy(self.ctx) }
    }
}

impl Gpu {
    /// `sign` of messages fed twice in pieces (blocking creation).  D224 is refused (capy_gpu.h: quirk Q7).
    pub fn sign_stream(&self, keys: &[&KeyPair], d: SecParam) -> Result<SignStream, OperationError> {
        let (pd, po) = pack(keys.iter().map(|k| k.priv_key.as_slice()));
        let mut h = std::ptr::null_mut();
        status(unsafe { capy_ed448_sign_stream_new(self.ctx, d as c_int, pd.as_ptr(), po.as_ptr(), keys.len() as u64, &mut h) })?;
        Ok(SignStream { ctx: self.ctx, h, n: keys.len() })
    }

    /// `sha3_decrypt` of ciphertexts fed twice in pieces; every nonce has `nonces[0].len()` bytes and every tag 64.
    pub fn sha3_decrypt_stream(&self, pws: &[&[u8]], nonces: &[&[u8]], tags: &[&[u8]], d: SecParam)
                               -> Result<DecryptStream, OperationError> {
        let n = pws.len();
        let nonce_len = nonces.first().map_or(0, |z| z.len());
        if nonces.len() != n || tags.len() != n || nonces.iter().any(|z| z.len() != nonce_len) || tags.iter().any(|t| t.len() != 64) {
            return Err(OperationError::SHA3DecryptionFailure);
        }
        let (pd, po) = pack(pws.iter().copied());
        let (zd, _) = pack(nonces.iter().copied());
        let (td, _) = pack(tags.iter().copied());
        let mut h = std::ptr::null_mut();
        status(unsafe {
            capy_sponge_decrypt_stream_new(self.ctx, d as c_int, CAPY_AE_SHA3, pd.as_ptr(), po.as_ptr(), zd.as_ptr(),
                                           nonce_len as u64, td.as_ptr(), n as u64, &mut h)
        })?;
        Ok(DecryptStream { ctx: self.ctx, h, n, key: false })
    }

    /// `key_decrypt` of ciphertexts fed twice in pieces; `asym_nonces[i]` is Z_i (112 bytes), every tag 56 bytes.
    pub fn key_decrypt_stream(&self, pws: &[&[u8]], asym_nonces: &[&[u8]], tags: &[&[u8]], d: SecParam)
                              -> Result<DecryptStream, OperationError> {
        let n = pws.len();
        if asym_nonces.len() != n || tags.len() != n || asym_nonces.iter().any(|z| z.len() != 112) || tags.iter().any(|t| t.len() != 56) {
            return Err(OperationError::KeyDecryptionError);
        }
        let (pd, po) = pack(pws.iter().copied());
        let (zd, _) = pack(asym_nonces.iter().copied());
        let (td, _) = pack(tags.iter().copied());
        let mut h = std::ptr::null_mut();
        status(unsafe {
            capy_ed448_key_decrypt_stream_new(self.ctx, d as c_int, pd.as_ptr(), po.as_ptr(), zd.as_ptr(), td.as_ptr(), n as u64,
                                              &mut h)
        })?;
        Ok(DecryptStream { ctx: self.ctx, h, n, key: true })
    }
}
