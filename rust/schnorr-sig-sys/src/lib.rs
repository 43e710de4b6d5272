//! Raw bindings to `include/schnorr_b200.h` and a minimal safe wrapper.
//!
//! Record layouts are the reference's own encodings, so the callers copy bytes, they do not convert:
//! signature 81 B = `Signature::to_bytes()`; public key 96 B = affine `x || y` limbs + one identity flag byte;
//! scalar 32 B little-endian; messages = one blob + `u64` offsets (`&[&[u8]]` flattened).
//! Verdict bytes: 0 `Ok(())`, 1 `InvalidPublicKey`, 2 `InvalidSignature`, 3 = input on which the reference panics.
#![allow(non_camel_case_types)]

use core::ffi::{c_char, c_int, c_uint, c_void};

#[repr(C)]
pub struct schnorr_b200_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct schnorr_b200_keyset {
    _private: [u8; 0],
}

pub const SCHNORR_B200_OK: c_int = 0;
pub const SCHNORR_B200_EARG: c_int = -1;
pub const SCHNORR_B200_ECUDA: c_int = -2;
pub const SCHNORR_B200_ENODEV: c_int = -3;

extern "C" {
    pub fn schnorr_b200_params_pinned() -> c_int;
    pub fn schnorr_b200_params_provenance() -> *const c_char;
    pub fn schnorr_b200_create(device: c_int, out: *mut *mut schnorr_b200_ctx) -> c_int;
    pub fn schnorr_b200_create_multi(devices: *const c_int, n_devices: c_int, out: *mut *mut schnorr_b200_ctx) -> c_int;
    pub fn schnorr_b200_device_count(ctx: *const schnorr_b200_ctx) -> c_int;
    pub fn schnorr_b200_destroy(ctx: *mut schnorr_b200_ctx);
    pub fn schnorr_b200_last_error(ctx: *const schnorr_b200_ctx) -> *const c_char;
    pub fn schnorr_b200_set_stream(ctx: *mut schnorr_b200_ctx, stream: *mut c_void) -> c_int;
    pub fn schnorr_b200_synchronize(ctx: *mut schnorr_b200_ctx) -> c_int;

    pub fn schnorr_b200_hash_messages(ctx: *mut schnorr_b200_ctx, n: usize, rx48: *const u8, pk96: *const u8,
        msgs: *const u8, msg_off: *const u64, digests: *mut u8) -> c_int;
    pub fn schnorr_b200_verify_many(ctx: *mut schnorr_b200_ctx, n: usize, sigs81: *const u8, pk96: *const u8,
        pk_inf: *const u8, msgs: *const u8, msg_off: *const u64, verdicts: *mut u8) -> c_int;
    pub fn schnorr_b200_verify_keyed_many(ctx: *mut schnorr_b200_ctx, n: usize, keyed130: *const u8, msgs: *const u8,
        msg_off: *const u64, verdicts: *mut u8) -> c_int;
    pub fn schnorr_b200_verify_batch(ctx: *mut schnorr_b200_ctx, n: usize, sigs81: *const u8, pk96: *const u8,
        pk_inf: *const u8, msgs: *const u8, msg_off: *const u64, rand32: *const u8, verdict: *mut c_int,
        lhs97: *mut u8, rhs97: *mut u8) -> c_int;
    pub fn schnorr_b200_locate_invalid(ctx: *mut schnorr_b200_ctx, n: usize, sigs81: *const u8, pk96: *const u8,
        pk_inf: *const u8, msgs: *const u8, msg_off: *const u64, rand32: *const u8, flags: *mut u8,
        n_bad: *mut u64) -> c_int;
    pub fn schnorr_b200_batch_randomizers(ctx: *mut schnorr_b200_ctx, n: usize, seed32: *const u8, first_index: u64,
        rand32: *mut u8) -> c_int;
    pub fn schnorr_b200_batch_randomizers_dev(ctx: *mut schnorr_b200_ctx, n: usize, seed32: *const u8, first_index: u64,
        rand32: *mut u8) -> c_int;
    pub fn schnorr_b200_verify_batch_seeded(ctx: *mut schnorr_b200_ctx, n: usize, sigs81: *const u8, pk96: *const u8,
        pk_inf: *const u8, msgs: *const u8, msg_off: *const u64, seed32: *const u8, verdict: *mut c_int,
        lhs97: *mut u8, rhs97: *mut u8) -> c_int;
    pub fn schnorr_b200_verify_batch_registered_seeded(ctx: *mut schnorr_b200_ctx, ks: *const schnorr_b200_keyset,
        n: usize, sigs81: *const u8, key_idx: *const u32, msgs: *const u8, msg_off: *const u64, seed32: *const u8,
        verdict: *mut c_int, lhs97: *mut u8, rhs97: *mut u8) -> c_int;
    pub fn schnorr_b200_verify_batch_keyed_seeded(ctx: *mut schnorr_b200_ctx, n: usize, keyed130: *const u8,
        msgs: *const u8, msg_off: *const u64, seed32: *const u8, verdict: *mut c_int, lhs97: *mut u8,
        rhs97: *mut u8) -> c_int;
    pub fn schnorr_b200_verify_batch_keyed_registered_seeded(ctx: *mut schnorr_b200_ctx, ks: *const schnorr_b200_keyset,
        n: usize, keyed130: *const u8, msgs: *const u8, msg_off: *const u64, seed32: *const u8, verdict: *mut c_int,
        lhs97: *mut u8, rhs97: *mut u8) -> c_int;
    pub fn schnorr_b200_locate_invalid_seeded(ctx: *mut schnorr_b200_ctx, n: usize, sigs81: *const u8, pk96: *const u8,
        pk_inf: *const u8, msgs: *const u8, msg_off: *const u64, seed32: *const u8, flags: *mut u8,
        n_bad: *mut u64) -> c_int;
    pub fn schnorr_b200_locate_invalid_registered_seeded(ctx: *mut schnorr_b200_ctx, ks: *const schnorr_b200_keyset,
        n: usize, sigs81: *const u8, key_idx: *const u32, msgs: *const u8, msg_off: *const u64, seed32: *const u8,
        flags: *mut u8, n_bad: *mut u64) -> c_int;
    pub fn schnorr_b200_locate_invalid_keyed_seeded(ctx: *mut schnorr_b200_ctx, n: usize, keyed130: *const u8,
        msgs: *const u8, msg_off: *const u64, seed32: *const u8, flags: *mut u8, n_bad: *mut u64) -> c_int;
    pub fn schnorr_b200_locate_invalid_keyed_registered_seeded(ctx: *mut schnorr_b200_ctx, ks: *const schnorr_b200_keyset,
        n: usize, keyed130: *const u8, msgs: *const u8, msg_off: *const u64, seed32: *const u8, flags: *mut u8,
        n_bad: *mut u64) -> c_int;
    pub fn schnorr_b200_keygen(ctx: *mut schnorr_b200_ctx, n: usize, sk32: *const u8, pk96: *mut u8, pk_inf: *mut u8) -> c_int;
    pub fn schnorr_b200_sign_many(ctx: *mut schnorr_b200_ctx, n: usize, sk32: *const u8, pk96: *const u8,
        pk_inf: *const u8, msgs: *const u8, msg_off: *const u64, nonce32: *const u8, sigs81: *mut u8) -> c_int;
    pub fn schnorr_b200_decompress(ctx: *mut schnorr_b200_ctx, n: usize, in49: *const u8, pk96: *mut u8,
        pk_inf: *mut u8, ok: *mut u8) -> c_int;
    pub fn schnorr_b200_compress(ctx: *mut schnorr_b200_ctx, n: usize, pk96: *const u8, pk_inf: *const u8,
        out49: *mut u8) -> c_int;
    pub fn schnorr_b200_derive_master_keys(ctx: *mut schnorr_b200_ctx, n: usize, seeds32: *const u8, xsk64: *mut u8,
        ok: *mut u8) -> c_int;
    pub fn schnorr_b200_derive_private_children(ctx: *mut schnorr_b200_ctx, n: usize, parent_xsk64: *const u8,
        indices: *const u32, children_xsk64: *mut u8, ok: *mut u8) -> c_int;
    pub fn schnorr_b200_derive_public_children(ctx: *mut schnorr_b200_ctx, n: usize, parent_xpk81: *const u8,
        indices: *const u32, children_xpk81: *mut u8, ok: *mut u8) -> c_int;
    pub fn schnorr_b200_set_dist_threshold(ctx: *mut schnorr_b200_ctx, max_signatures: usize) -> c_int;
    pub fn schnorr_b200_set_one_threshold(ctx: *mut schnorr_b200_ctx, max_signatures: usize) -> c_int;
    pub fn schnorr_b200_set_batch_small_threshold(ctx: *mut schnorr_b200_ctx, max_signatures: usize) -> c_int;
    pub fn schnorr_b200_set_msm_geometry(ctx: *mut schnorr_b200_ctx, window_bits: c_int, segment_len: c_uint) -> c_int;
}

/// Flattened `&[&[u8]]`: the blob and its `n + 1` offsets.
pub fn pack_messages(messages: &[&[u8]]) -> (Vec<u8>, Vec<u64>) {
    let mut off = Vec::with_capacity(messages.len() + 1);
    let mut blob = Vec::with_capacity(messages.iter().map(|m| m.len()).sum());
    off.push(0u64);
    for m in messages {
        blob.extend_from_slice(m);
        off.push(blob.len() as u64);
    }
    (blob, off)
}

/// One context (single- or multi-device).  The C context is single-owner: keep one `Engine` per thread, or guard it.
pub struct Engine(*mut schnorr_b200_ctx);
unsafe impl Send for Engine {}

impl Engine {
    /// `devices`: CUDA device indices; several entries give a multi-device context whose calls are sharded.
    pub fn new(devices: &[i32]) -> Result<Self, i32> {
        let mut p = core::ptr::null_mut();
        let rc = unsafe { schnorr_b200_create_multi(devices.as_ptr(), devices.len() as c_int, &mut p) };
        if rc == SCHNORR_B200_OK { Ok(Engine(p)) } else { Err(rc) }
    }

    /// `true` once the compiled-in constants were dumped from the real `cheetah` / `hash` crates.
    pub fn params_pinned() -> bool {
        unsafe { schnorr_b200_params_pinned() != 0 }
    }

    fn check(&self, rc: c_int, what: &str) {
        if rc != SCHNORR_B200_OK {
            let msg = unsafe { core::ffi::CStr::from_ptr(schnorr_b200_last_error(self.0)) };
            panic!("{what} failed ({rc}): {}", msg.to_string_lossy());
        }
    }

    pub fn verify_many(&self, sigs: &[[u8; 81]], pks: &[[u8; 96]], pk_inf: &[u8], messages: &[&[u8]]) -> Vec<u8> {
        assert!(sigs.len() == pks.len() && pk_inf.len() == sigs.len() && messages.len() == sigs.len());
        let (blob, off) = pack_messages(messages);
        let mut v = vec![255u8; sigs.len()];
        let rc = unsafe {
            schnorr_b200_verify_many(self.0, sigs.len(), sigs.as_ptr().cast(), pks.as_ptr().cast(), pk_inf.as_ptr(),
                                     blob.as_ptr(), off.as_ptr(), v.as_mut_ptr())
        };
        self.check(rc, "schnorr_b200_verify_many");
        v
    }

    /// Returns the batch verdict (0 / 2 / 3).
    pub fn verify_batch(&self, sigs: &[[u8; 81]], pks: &[[u8; 96]], pk_inf: &[u8], messages: &[&[u8]], rand: &[[u8; 32]]) -> u8 {
        assert!(sigs.len() == pks.len() && rand.len() == sigs.len() && messages.len() == sigs.len());
        let (blob, off) = pack_messages(messages);
        let mut verdict: c_int = -1;
        let rc = unsafe {
            schnorr_b200_verify_batch(self.0, sigs.len(), sigs.as_ptr().cast(), pks.as_ptr().cast(), pk_inf.as_ptr(),
                                      blob.as_ptr(), off.as_ptr(), rand.as_ptr().cast(), &mut verdict,
                                      core::ptr::null_mut(), core::ptr::null_mut())
        };
        self.check(rc, "schnorr_b200_verify_batch");
        verdict as u8
    }

    /// `verify_batch` with randomisers `0 .. n` generated on the device from a 32-byte seed; returns the verdict.
    pub fn verify_batch_seeded(&self, sigs: &[[u8; 81]], pks: &[[u8; 96]], pk_inf: &[u8], messages: &[&[u8]],
                               seed: &[u8; 32]) -> u8 {
        assert!(sigs.len() == pks.len() && messages.len() == sigs.len());
        let (blob, off) = pack_messages(messages);
        let mut verdict: c_int = -1;
        let rc = unsafe {
            schnorr_b200_verify_batch_seeded(self.0, sigs.len(), sigs.as_ptr().cast(), pks.as_ptr().cast(), pk_inf.as_ptr(),
                                             blob.as_ptr(), off.as_ptr(), seed.as_ptr(), &mut verdict,
                                             core::ptr::null_mut(), core::ptr::null_mut())
        };
        self.check(rc, "schnorr_b200_verify_batch_seeded");
        verdict as u8
    }

    /// Randomisers `first .. first + n` of a seed: the `rand` that `verify_batch_seeded` used for `first = 0`.
    pub fn batch_randomizers(&self, n: usize, seed: &[u8; 32], first: u64) -> Vec<[u8; 32]> {
        let mut rand = vec![[0u8; 32]; n];
        let rc = unsafe { schnorr_b200_batch_randomizers(self.0, n, seed.as_ptr(), first, rand.as_mut_ptr().cast()) };
        self.check(rc, "schnorr_b200_batch_randomizers");
        rand
    }

    /// Per-item flags of a failed batch, batch semantics (0 clean, 2 culprit, 3 malformed).
    pub fn locate_invalid(&self, sigs: &[[u8; 81]], pks: &[[u8; 96]], pk_inf: &[u8], messages: &[&[u8]], rand: &[[u8; 32]]) -> Vec<u8> {
        let (blob, off) = pack_messages(messages);
        let mut flags = vec![0u8; sigs.len()];
        let rc = unsafe {
            schnorr_b200_locate_invalid(self.0, sigs.len(), sigs.as_ptr().cast(), pks.as_ptr().cast(), pk_inf.as_ptr(),
                                        blob.as_ptr(), off.as_ptr(), rand.as_ptr().cast(), flags.as_mut_ptr(),
                                        core::ptr::null_mut())
        };
        self.check(rc, "schnorr_b200_locate_invalid");
        flags
    }

    /// `locate_invalid` with randomisers `0 .. n` generated on the devices from a 32-byte seed: the flags of a failed
    /// `verify_batch_seeded`.
    pub fn locate_invalid_seeded(&self, sigs: &[[u8; 81]], pks: &[[u8; 96]], pk_inf: &[u8], messages: &[&[u8]],
                                 seed: &[u8; 32]) -> Vec<u8> {
        let (blob, off) = pack_messages(messages);
        let mut flags = vec![0u8; sigs.len()];
        let rc = unsafe {
            schnorr_b200_locate_invalid_seeded(self.0, sigs.len(), sigs.as_ptr().cast(), pks.as_ptr().cast(),
                                               pk_inf.as_ptr(), blob.as_ptr(), off.as_ptr(), seed.as_ptr(),
                                               flags.as_mut_ptr(), core::ptr::null_mut())
        };
        self.check(rc, "schnorr_b200_locate_invalid_seeded");
        flags
    }

    pub fn hash_messages(&self, rx: &[[u8; 48]], pks: &[[u8; 96]], messages: &[&[u8]]) -> Vec<[u8; 32]> {
        let (blob, off) = pack_messages(messages);
        let mut d = vec![[0u8; 32]; rx.len()];
        let rc = unsafe {
            schnorr_b200_hash_messages(self.0, rx.len(), rx.as_ptr().cast(), pks.as_ptr().cast(), blob.as_ptr(),
                                       off.as_ptr(), d.as_mut_ptr().cast())
        };
        self.check(rc, "schnorr_b200_hash_messages");
        d
    }
}

impl Drop for Engine {
    fn drop(&mut self) {
        unsafe { schnorr_b200_destroy(self.0) }
    }
}
