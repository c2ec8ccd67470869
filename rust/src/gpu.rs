// Safe wrappers over the C ABI: the drop-in surface of the reference crate's verify path (feature `gpu`).
//
//   crate::gpu::GpuVerifier           one context over one or more B200s; the batch entry points
//   crate::gpu::global()              the process-wide verifier behind the scalar drop-ins
//   crate::gpu::verify_single(..) ..  what PublicKey::verify / PublicKeyDouble::verify / PublicKeyVarGen::verify call when the
//                                     feature is on (patches/verify_methods.patch), so their signatures stay the reference's
//
// NOT compiled in this repository's environment (no cargo / rustc in the image); written against include/jjschnorr_b200.h,
// which is compiled and tested.  tests/test_abi.py checks that every host entry point of the header is wrapped here.
#![cfg(feature = "gpu")]

extern crate std;

use core::ffi::c_int;
use std::ffi::CStr;
use std::ptr;
use std::string::String;
use std::sync::{Mutex, MutexGuard, OnceLock};
use std::vec::Vec;

use dusk_bls12_381::BlsScalar;
use dusk_bytes::Serializable;
use dusk_jubjub::JubJubExtended;

use crate::{Error, PublicKey, PublicKeyDouble, PublicKeyVarGen, Signature, SignatureDouble, SignatureVarGen};

#[path = "ffi.rs"]
mod ffi;

/// Owns a `jjs_ctx`.  One host thread at a time per context (the header's threading rule), hence `&mut self` everywhere.
pub struct GpuVerifier {
    ctx: *mut ffi::jjs_ctx,
}
unsafe impl Send for GpuVerifier {}

fn status_to_result(status: u8) -> Result<(), Error> {
    match status {
        ffi::JJS_OK => Ok(()),
        ffi::JJS_INVALID_SIGNATURE => Err(Error::InvalidSignature), // src/error.rs:17
        ffi::JJS_INVALID_POINT => Err(Error::InvalidPoint),         // src/error.rs:19
        _ => Err(Error::BytesError(dusk_bytes::Error::InvalidData)), // src/error.rs:15
    }
}

fn unpack(words: &[u32], n: usize) -> Vec<bool> {
    (0..n).map(|i| (words[i / 32] >> (i % 32)) & 1 == 1).collect()
}

/// `to_bytes()` of every field of a batch into three contiguous arrays (what the C ABI takes).
fn wire<K, S, const KN: usize, const SN: usize>(items: &[(K, S, BlsScalar)]) -> (Vec<u8>, Vec<u8>, Vec<u8>)
where
    K: Serializable<KN>,
    S: Serializable<SN>,
{
    let n = items.len();
    let (mut pk, mut sig, mut msg) = (Vec::with_capacity(KN * n), Vec::with_capacity(SN * n), Vec::with_capacity(32 * n));
    for (k, s, m) in items {
        pk.extend_from_slice(&k.to_bytes()); // src/keys/public.rs:83-85 (one field inversion per point on the CPU)
        sig.extend_from_slice(&s.to_bytes()); // src/signatures.rs:104-109
        msg.extend_from_slice(&m.to_bytes());
    }
    (pk, sig, msg)
}

/// The five coordinates of a JubJubExtended exactly as they sit in memory (Montgomery limbs): no arithmetic on the CPU.
fn push_point(buf: &mut Vec<u8>, p: &JubJubExtended) {
    for c in [p.get_u(), p.get_v(), p.get_z(), p.get_t1(), p.get_t2()] {
        for limb in c.0 {
            buf.extend_from_slice(&limb.to_le_bytes());
        }
    }
}

impl GpuVerifier {
    /// `devices`: CUDA ordinals.  Batches are split into contiguous shards, one host thread and one set of streams per GPU,
    /// no collective.  Fails (no CPU fallback) when no sm_100a device is usable.
    pub fn new(devices: &[i32]) -> Result<Self, String> {
        let mut ctx = ptr::null_mut();
        let rc = unsafe { ffi::jjs_init(devices.as_ptr(), devices.len() as i32, &mut ctx) };
        Self::from_init(rc, ctx)
    }

    /// A verifier that holds at most `device_memory_limit` bytes of device memory on each of `devices` (jjs_init_limited): the
    /// library picks the fastest configuration that fits.  Fails when even the smallest one (about 40 MB) does not.
    pub fn with_memory_limit(devices: &[i32], device_memory_limit: usize) -> Result<Self, String> {
        let mut ctx = ptr::null_mut();
        let rc = unsafe { ffi::jjs_init_limited(devices.as_ptr(), devices.len() as i32, device_memory_limit, &mut ctx) };
        Self::from_init(rc, ctx)
    }

    fn from_init(rc: i32, ctx: *mut ffi::jjs_ctx) -> Result<Self, String> {
        if rc != 0 {
            let msg = if ctx.is_null() {
                String::from("jjs_init: allocation failed")
            } else {
                unsafe { CStr::from_ptr(ffi::jjs_last_error(ctx)) }.to_string_lossy().into_owned()
            };
            unsafe { ffi::jjs_destroy(ctx) };
            return Err(msg);
        }
        Ok(Self { ctx })
    }

    fn check(&self, rc: i32, what: &str) {
        if rc != 0 {
            let msg = unsafe { CStr::from_ptr(ffi::jjs_last_error(self.ctx)) }.to_string_lossy().into_owned();
            panic!("{what} failed ({rc}): {msg}");
        }
    }

    // ---- single: PublicKey::verify (src/keys/public.rs:114-135) -------------------------------------------------------
    /// NEW: verify_batch(&[(PublicKey, Signature, BlsScalar)]) -> Vec<bool>, bit-exact with
    /// `items.iter().map(|(pk, sig, m)| pk.verify(sig, *m).is_ok())`; the accept bits are packed on the GPU.
    pub fn verify_batch(&mut self, items: &[(PublicKey, Signature, BlsScalar)]) -> Vec<bool> {
        let n = items.len();
        let (pk, sig, msg) = wire::<_, _, 32, 64>(items);
        let mut words = vec![0u32; (n + 31) / 32];
        let rc = unsafe { ffi::jjs_verify_batch(self.ctx, pk.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, words.as_mut_ptr()) };
        self.check(rc, "jjs_verify_batch");
        unpack(&words, n)
    }

    /// Same, keeping the reference's error variant per item.
    pub fn verify_batch_status(&mut self, items: &[(PublicKey, Signature, BlsScalar)]) -> Vec<Result<(), Error>> {
        let n = items.len();
        let (pk, sig, msg) = wire::<_, _, 32, 64>(items);
        let mut status = vec![0u8; n];
        let rc = unsafe { ffi::jjs_verify_single(self.ctx, pk.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, status.as_mut_ptr(), ptr::null_mut()) };
        self.check(rc, "jjs_verify_single");
        status.into_iter().map(status_to_result).collect()
    }

    /// NEW: `items.iter().all(|(pk, sig, m)| pk.verify(sig, *m).is_ok())` by one random linear combination of all the equations
    /// (jjs_verify_all, fresh secret weights from the operating system): a batch with a failing item passes with probability at
    /// most 2^-128.  No per-item answer: call verify_batch to find the failing items.
    pub fn verify_all(&mut self, items: &[(PublicKey, Signature, BlsScalar)]) -> bool {
        let n = items.len();
        let (pk, sig, msg) = wire::<_, _, 32, 64>(items);
        let mut ok: c_int = 0;
        let rc = unsafe { ffi::jjs_verify_all(self.ctx, ffi::JJS_KIND_SINGLE, pk.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, ptr::null(), &mut ok) };
        self.check(rc, "jjs_verify_all");
        ok == 1
    }

    /// The same for double items.
    pub fn verify_all_double(&mut self, items: &[(PublicKeyDouble, SignatureDouble, BlsScalar)]) -> bool {
        let n = items.len();
        let (pk, sig, msg) = wire::<_, _, 64, 96>(items);
        let mut ok: c_int = 0;
        let rc = unsafe { ffi::jjs_verify_all(self.ctx, ffi::JJS_KIND_DOUBLE, pk.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, ptr::null(), &mut ok) };
        self.check(rc, "jjs_verify_all");
        ok == 1
    }

    // ---- double: PublicKeyDouble::verify (src/keys/public/double.rs:86-117) --------------------------------------------
    pub fn verify_batch_double(&mut self, items: &[(PublicKeyDouble, SignatureDouble, BlsScalar)]) -> Vec<bool> {
        let n = items.len();
        let (pk, sig, msg) = wire::<_, _, 64, 96>(items);
        let mut words = vec![0u32; (n + 31) / 32];
        let rc = unsafe { ffi::jjs_verify_batch_double(self.ctx, pk.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, words.as_mut_ptr()) };
        self.check(rc, "jjs_verify_batch_double");
        unpack(&words, n)
    }

    pub fn verify_batch_double_status(&mut self, items: &[(PublicKeyDouble, SignatureDouble, BlsScalar)]) -> Vec<Result<(), Error>> {
        let n = items.len();
        let (pk, sig, msg) = wire::<_, _, 64, 96>(items);
        let mut status = vec![0u8; n];
        let rc = unsafe { ffi::jjs_verify_double(self.ctx, pk.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, status.as_mut_ptr(), ptr::null_mut()) };
        self.check(rc, "jjs_verify_double");
        status.into_iter().map(status_to_result).collect()
    }

    // ---- variable generator: PublicKeyVarGen::verify (src/keys/public/var_gen.rs:107-133) ------------------------------
    pub fn verify_batch_var_gen(&mut self, items: &[(PublicKeyVarGen, SignatureVarGen, BlsScalar)]) -> Vec<bool> {
        let n = items.len();
        let (pk, sig, msg) = wire::<_, _, 64, 64>(items);
        let mut words = vec![0u32; (n + 31) / 32];
        let rc = unsafe { ffi::jjs_verify_batch_vargen(self.ctx, pk.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, words.as_mut_ptr()) };
        self.check(rc, "jjs_verify_batch_vargen");
        unpack(&words, n)
    }

    pub fn verify_batch_var_gen_status(&mut self, items: &[(PublicKeyVarGen, SignatureVarGen, BlsScalar)]) -> Vec<Result<(), Error>> {
        let n = items.len();
        let (pk, sig, msg) = wire::<_, _, 64, 64>(items);
        let mut status = vec![0u8; n];
        let rc = unsafe { ffi::jjs_verify_vargen(self.ctx, pk.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, status.as_mut_ptr(), ptr::null_mut()) };
        self.check(rc, "jjs_verify_vargen");
        status.into_iter().map(status_to_result).collect()
    }

    // ---- aggregate key: multisig::aggregate_pk(..).verify(..) (src/multisig.rs:154-156, 393-429) ----------------------
    fn ragged(items: &[(&[PublicKey], Signature, BlsScalar)]) -> (Vec<u8>, Vec<u32>, Vec<u8>, Vec<u8>) {
        let n = items.len();
        let (mut pks, mut offsets) = (Vec::new(), Vec::with_capacity(n + 1));
        let (mut sig, mut msg) = (Vec::with_capacity(64 * n), Vec::with_capacity(32 * n));
        offsets.push(0u32);
        for (signers, s, m) in items {
            for pk in signers.iter() {
                pks.extend_from_slice(&pk.to_bytes());
            }
            offsets.push((pks.len() / 32) as u32);
            sig.extend_from_slice(&s.to_bytes());
            msg.extend_from_slice(&m.to_bytes());
        }
        (pks, offsets, sig, msg)
    }

    /// `aggregate_pk(signers).verify(sig, msg).is_ok()` per item; any number of signers per item.
    pub fn verify_batch_aggregate(&mut self, items: &[(&[PublicKey], Signature, BlsScalar)]) -> Vec<bool> {
        let n = items.len();
        let (pks, offsets, sig, msg) = Self::ragged(items);
        let mut words = vec![0u32; (n + 31) / 32];
        let rc = unsafe {
            ffi::jjs_verify_batch_aggregate(self.ctx, pks.as_ptr(), offsets.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, words.as_mut_ptr())
        };
        self.check(rc, "jjs_verify_batch_aggregate");
        unpack(&words, n)
    }

    /// Per item: the verify result and `aggregate_pk(signers).to_bytes()` (all zero when a signer key does not decode).
    pub fn verify_batch_aggregate_status(&mut self, items: &[(&[PublicKey], Signature, BlsScalar)]) -> Vec<(Result<(), Error>, [u8; 32])> {
        let n = items.len();
        let (pks, offsets, sig, msg) = Self::ragged(items);
        let (mut status, mut agg) = (vec![0u8; n], vec![0u8; 32 * n]);
        let rc = unsafe {
            ffi::jjs_verify_aggregate(self.ctx, pks.as_ptr(), offsets.as_ptr(), sig.as_ptr(), msg.as_ptr(), n, status.as_mut_ptr(),
                                      ptr::null_mut(), agg.as_mut_ptr())
        };
        self.check(rc, "jjs_verify_aggregate");
        (0..n).map(|i| {
            let mut key = [0u8; 32];
            key.copy_from_slice(&agg[32 * i..32 * i + 32]);
            (status_to_result(status[i]), key)
        }).collect()
    }

    // ---- typed inputs: no to_bytes(), the GPU normalises the points (jjs_verify_ext) ----------------------------------
    pub fn verify_batch_typed(&mut self, items: &[(PublicKey, Signature, BlsScalar)]) -> Vec<Result<(), Error>> {
        let n = items.len();
        let (mut pts, mut u, mut msg) = (Vec::with_capacity(320 * n), Vec::with_capacity(32 * n), Vec::with_capacity(32 * n));
        for (pk, sig, m) in items {
            push_point(&mut pts, pk.as_ref()); // src/keys/public.rs:74-78
            push_point(&mut pts, sig.R()); // src/signatures.rs:75-77
            u.extend_from_slice(&sig.u().to_bytes()); // one Montgomery reduction, no inversion
            msg.extend_from_slice(&m.to_bytes());
        }
        self.run_typed(0, &pts, &u, &msg, n)
    }

    pub fn verify_batch_double_typed(&mut self, items: &[(PublicKeyDouble, SignatureDouble, BlsScalar)]) -> Vec<Result<(), Error>> {
        let n = items.len();
        let (mut pts, mut u, mut msg) = (Vec::with_capacity(640 * n), Vec::with_capacity(32 * n), Vec::with_capacity(32 * n));
        for (pk, sig, m) in items {
            push_point(&mut pts, pk.pk()); // src/keys/public/double.rs:60-62
            push_point(&mut pts, pk.pk_prime());
            push_point(&mut pts, sig.R()); // src/signatures/double.rs:80-88
            push_point(&mut pts, sig.R_prime());
            u.extend_from_slice(&sig.u().to_bytes());
            msg.extend_from_slice(&m.to_bytes());
        }
        self.run_typed(1, &pts, &u, &msg, n)
    }

    pub fn verify_batch_var_gen_typed(&mut self, items: &[(PublicKeyVarGen, SignatureVarGen, BlsScalar)]) -> Vec<Result<(), Error>> {
        let n = items.len();
        let (mut pts, mut u, mut msg) = (Vec::with_capacity(480 * n), Vec::with_capacity(32 * n), Vec::with_capacity(32 * n));
        for (pk, sig, m) in items {
            push_point(&mut pts, pk.public_key()); // src/keys/public/var_gen.rs:83-90
            push_point(&mut pts, pk.generator());
            push_point(&mut pts, sig.R()); // src/signatures/var_gen.rs:69-71
            u.extend_from_slice(&sig.u().to_bytes());
            msg.extend_from_slice(&m.to_bytes());
        }
        self.run_typed(2, &pts, &u, &msg, n)
    }

    fn run_typed(&mut self, variant: i32, pts: &[u8], u: &[u8], msg: &[u8], n: usize) -> Vec<Result<(), Error>> {
        let mut status = vec![0u8; n];
        let rc = unsafe { ffi::jjs_verify_ext(self.ctx, variant, pts.as_ptr(), u.as_ptr(), msg.as_ptr(), n, status.as_mut_ptr(), ptr::null_mut()) };
        self.check(rc, "jjs_verify_ext");
        status.into_iter().map(status_to_result).collect()
    }

    // ---- several kinds in one call (BASELINE configs[3] / [4]): the library balances them over its devices ---------------
    pub fn verify_mixed(&mut self, singles: &[(PublicKey, Signature, BlsScalar)], doubles: &[(PublicKeyDouble, SignatureDouble, BlsScalar)],
                        var_gens: &[(PublicKeyVarGen, SignatureVarGen, BlsScalar)]) -> (Vec<bool>, Vec<bool>, Vec<bool>) {
        let (a, b, c) = (wire::<_, _, 32, 64>(singles), wire::<_, _, 64, 96>(doubles), wire::<_, _, 64, 64>(var_gens));
        let (na, nb, nc) = (singles.len(), doubles.len(), var_gens.len());
        let (mut wa, mut wb, mut wc) = (vec![0u32; (na + 31) / 32], vec![0u32; (nb + 31) / 32], vec![0u32; (nc + 31) / 32]);
        let part = |kind, w: &(Vec<u8>, Vec<u8>, Vec<u8>), n, words: &mut Vec<u32>| ffi::jjs_part {
            kind, pk: w.0.as_ptr(), offsets: ptr::null(), sig: w.1.as_ptr(), msg32: w.2.as_ptr(), n,
            status: ptr::null_mut(), c32: ptr::null_mut(), aggpk32: ptr::null_mut(), accept_bitmap: words.as_mut_ptr(),
        };
        let parts = [part(ffi::JJS_KIND_SINGLE, &a, na, &mut wa), part(ffi::JJS_KIND_DOUBLE, &b, nb, &mut wb),
                     part(ffi::JJS_KIND_VARGEN, &c, nc, &mut wc)];
        let rc = unsafe { ffi::jjs_verify_mixed(self.ctx, parts.as_ptr(), parts.len()) };
        self.check(rc, "jjs_verify_mixed");
        (unpack(&wa, na), unpack(&wb, nb), unpack(&wc, nc))
    }

    /// NEW: whether every item of the three lists verifies, by one random linear combination over all of them
    /// (jjs_verify_all_mixed, fresh secret weights): a batch with a failing item passes with probability at most 2^-128.
    pub fn verify_all_mixed(&mut self, singles: &[(PublicKey, Signature, BlsScalar)], doubles: &[(PublicKeyDouble, SignatureDouble, BlsScalar)],
                            var_gens: &[(PublicKeyVarGen, SignatureVarGen, BlsScalar)]) -> bool {
        let (a, b, c) = (wire::<_, _, 32, 64>(singles), wire::<_, _, 64, 96>(doubles), wire::<_, _, 64, 64>(var_gens));
        let part = |kind, w: &(Vec<u8>, Vec<u8>, Vec<u8>), n| ffi::jjs_part {
            kind, pk: w.0.as_ptr(), offsets: ptr::null(), sig: w.1.as_ptr(), msg32: w.2.as_ptr(), n,
            status: ptr::null_mut(), c32: ptr::null_mut(), aggpk32: ptr::null_mut(), accept_bitmap: ptr::null_mut(),
        };
        let parts = [part(ffi::JJS_KIND_SINGLE, &a, singles.len()), part(ffi::JJS_KIND_DOUBLE, &b, doubles.len()),
                     part(ffi::JJS_KIND_VARGEN, &c, var_gens.len())];
        let mut ok: c_int = 0;
        let rc = unsafe { ffi::jjs_verify_all_mixed(self.ctx, parts.as_ptr(), parts.len(), ptr::null(), &mut ok) };
        self.check(rc, "jjs_verify_all_mixed");
        ok == 1
    }

    /// NEW: verify_mixed's per-item answers by one random linear combination per group of consecutive items, the per-item
    /// equations running only in groups whose combination fails (jjs_verify_grouped, fresh secret weights): a failing item is
    /// reported valid with probability at most 2^-128.
    pub fn verify_grouped(&mut self, singles: &[(PublicKey, Signature, BlsScalar)], doubles: &[(PublicKeyDouble, SignatureDouble, BlsScalar)],
                          var_gens: &[(PublicKeyVarGen, SignatureVarGen, BlsScalar)]) -> (Vec<bool>, Vec<bool>, Vec<bool>) {
        let (a, b, c) = (wire::<_, _, 32, 64>(singles), wire::<_, _, 64, 96>(doubles), wire::<_, _, 64, 64>(var_gens));
        let (na, nb, nc) = (singles.len(), doubles.len(), var_gens.len());
        let (mut wa, mut wb, mut wc) = (vec![0u32; (na + 31) / 32], vec![0u32; (nb + 31) / 32], vec![0u32; (nc + 31) / 32]);
        let part = |kind, w: &(Vec<u8>, Vec<u8>, Vec<u8>), n, words: &mut Vec<u32>| ffi::jjs_part {
            kind, pk: w.0.as_ptr(), offsets: ptr::null(), sig: w.1.as_ptr(), msg32: w.2.as_ptr(), n,
            status: ptr::null_mut(), c32: ptr::null_mut(), aggpk32: ptr::null_mut(), accept_bitmap: words.as_mut_ptr(),
        };
        let parts = [part(ffi::JJS_KIND_SINGLE, &a, na, &mut wa), part(ffi::JJS_KIND_DOUBLE, &b, nb, &mut wb),
                     part(ffi::JJS_KIND_VARGEN, &c, nc, &mut wc)];
        let rc = unsafe { ffi::jjs_verify_grouped(self.ctx, parts.as_ptr(), parts.len(), ptr::null(), ptr::null_mut()) };
        self.check(rc, "jjs_verify_grouped");
        (unpack(&wa, na), unpack(&wb, nb), unpack(&wc, nc))
    }
}

impl Drop for GpuVerifier {
    fn drop(&mut self) {
        unsafe { ffi::jjs_destroy(self.ctx) }
    }
}

// ---- the process-wide verifier behind the scalar drop-ins ------------------------------------------------------------------
static GLOBAL: OnceLock<Mutex<GpuVerifier>> = OnceLock::new();

/// The verifier the scalar methods use: created on first use over the devices named by `JJS_B200_DEVICES` ("0,1,2,..",
/// default "0"), holding at most `JJS_B200_MEMORY_LIMIT` bytes of device memory on each when that is set (else the full-size
/// context of `GpuVerifier::new`).  There is no CPU fallback: without a usable sm_100a device this panics with the library's message.
pub fn global() -> MutexGuard<'static, GpuVerifier> {
    GLOBAL
        .get_or_init(|| {
            let spec = std::env::var("JJS_B200_DEVICES").unwrap_or_else(|_| String::from("0"));
            let devices: Vec<i32> = spec.split(',').filter_map(|d| d.trim().parse().ok()).collect();
            let verifier = match std::env::var("JJS_B200_MEMORY_LIMIT") {
                Ok(limit) => {
                    let bytes: usize = limit.trim().parse().expect("JJS_B200_MEMORY_LIMIT: a number of bytes");
                    GpuVerifier::with_memory_limit(&devices, bytes)
                }
                Err(_) => GpuVerifier::new(&devices),
            };
            Mutex::new(verifier.expect("jubjub-schnorr gpu feature: no usable B200"))
        })
        .lock()
        .expect("gpu verifier poisoned")
}

/// Body of `PublicKey::verify(&self, &Signature, BlsScalar)` with the `gpu` feature (patches/verify_methods.patch).
pub fn verify_single(pk: &PublicKey, sig: &Signature, message: BlsScalar) -> Result<(), Error> {
    global().verify_batch_status(&[(*pk, *sig, message)]).pop().unwrap()
}
/// Body of `PublicKeyDouble::verify(&self, &SignatureDouble, BlsScalar)`.
pub fn verify_double(pk: &PublicKeyDouble, sig: &SignatureDouble, message: BlsScalar) -> Result<(), Error> {
    global().verify_batch_double_status(&[(*pk, *sig, message)]).pop().unwrap()
}
/// Body of `PublicKeyVarGen::verify(&self, &SignatureVarGen, BlsScalar)`.
pub fn verify_var_gen(pk: &PublicKeyVarGen, sig: &SignatureVarGen, message: BlsScalar) -> Result<(), Error> {
    global().verify_batch_var_gen_status(&[(*pk, *sig, message)]).pop().unwrap()
}
/// `multisig::aggregate_pk(signers)` followed by `.verify(sig, message)` in one device round trip.
pub fn verify_aggregate(signers: &[PublicKey], sig: &Signature, message: BlsScalar) -> Result<(), Error> {
    global().verify_batch_aggregate_status(&[(signers, *sig, message)]).pop().unwrap().0
}
/// NEW in the crate's public API: `verify_batch(&[(PublicKey, Signature, BlsScalar)]) -> Vec<bool>`.
pub fn verify_batch(items: &[(PublicKey, Signature, BlsScalar)]) -> Vec<bool> {
    global().verify_batch(items)
}
