// Raw bindings of include/jjschnorr_b200.h -- one declaration per exported function, in the header's order.
// tests/test_abi.py holds every declaration against the C header (names, parameter counts, pointer-ness, constness,
// integer widths, the status codes and the layout of jjs_part).  NOT compiled in this repository's environment.
#![allow(non_camel_case_types, dead_code)]
use core::ffi::{c_char, c_int, c_void};

#[repr(C)]
pub struct jjs_ctx {
    _private: [u8; 0],
}

pub const JJS_OK: u8 = 0; // Ok(())
pub const JJS_INVALID_SIGNATURE: u8 = 1; // Error::InvalidSignature   src/error.rs:17
pub const JJS_INVALID_POINT: u8 = 2; // Error::InvalidPoint       src/error.rs:19
pub const JJS_BYTES_ERROR: u8 = 3; // Error::BytesError(_)      src/error.rs:15
pub const JJS_INVALID_MULTISIG_TRANSCRIPT: u8 = 4; // Error::InvalidMultisigTranscript
pub const JJS_INVALID_MULTISIG_SHARE: u8 = 5; // Error::InvalidMultisigShare(index)

pub const JJS_KIND_SINGLE: c_int = 0;
pub const JJS_KIND_DOUBLE: c_int = 1;
pub const JJS_KIND_VARGEN: c_int = 2;
pub const JJS_KIND_AGGREGATE: c_int = 3;

/// One homogeneous batch of a `jjs_verify_mixed` call.
#[repr(C)]
pub struct jjs_part {
    pub kind: c_int,
    pub pk: *const u8,
    pub offsets: *const u32,
    pub sig: *const u8,
    pub msg32: *const u8,
    pub n: usize,
    pub status: *mut u8,
    pub c32: *mut u8,
    pub aggpk32: *mut u8,
    pub accept_bitmap: *mut u32,
}

extern "C" {
    pub fn jjs_init(devices: *const c_int, n_devices: c_int, out: *mut *mut jjs_ctx) -> c_int;
    // a context that never holds more than device_memory_limit bytes on any of its devices
    pub fn jjs_init_limited(devices: *const c_int, n_devices: c_int, device_memory_limit: usize, out: *mut *mut jjs_ctx) -> c_int;
    pub fn jjs_memory_info(ctx: *const jjs_ctx, device_index: c_int, bytes_held: *mut u64, fb_window_bits: *mut c_int,
                           items_in_flight: *mut u64) -> c_int;
    pub fn jjs_destroy(ctx: *mut jjs_ctx);
    pub fn jjs_last_error(ctx: *const jjs_ctx) -> *const c_char;
    pub fn jjs_device_count(ctx: *const jjs_ctx) -> c_int;
    // PublicKey::verify                      src/keys/public.rs:114-135
    pub fn jjs_verify_single(ctx: *mut jjs_ctx, pk32: *const u8, sig64: *const u8, msg32: *const u8, n: usize,
                             status: *mut u8, c32_or_null: *mut u8) -> c_int;
    // NEW verify_batch -> packed accept bitmap ((n + 31) / 32 words, bit i % 32 of word i / 32)
    pub fn jjs_verify_batch(ctx: *mut jjs_ctx, pk32: *const u8, sig64: *const u8, msg32: *const u8, n: usize,
                            accept_bitmap: *mut u32) -> c_int;
    pub fn jjs_verify_batch_double(ctx: *mut jjs_ctx, pk64: *const u8, sig96: *const u8, msg32: *const u8, n: usize,
                                   accept_bitmap: *mut u32) -> c_int;
    pub fn jjs_verify_batch_vargen(ctx: *mut jjs_ctx, pk64: *const u8, sig64: *const u8, msg32: *const u8, n: usize,
                                   accept_bitmap: *mut u32) -> c_int;
    pub fn jjs_verify_batch_aggregate(ctx: *mut jjs_ctx, pks32: *const u8, offsets: *const u32, sig64: *const u8,
                                      msg32: *const u8, n: usize, accept_bitmap: *mut u32) -> c_int;
    // PublicKeyDouble::verify                src/keys/public/double.rs:86-117
    pub fn jjs_verify_double(ctx: *mut jjs_ctx, pk64: *const u8, sig96: *const u8, msg32: *const u8, n: usize,
                             status: *mut u8, c32_or_null: *mut u8) -> c_int;
    // PublicKeyVarGen::verify                src/keys/public/var_gen.rs:107-133
    pub fn jjs_verify_vargen(ctx: *mut jjs_ctx, pk64: *const u8, sig64: *const u8, msg32: *const u8, n: usize,
                             status: *mut u8, c32_or_null: *mut u8) -> c_int;
    // multisig::aggregate_pk(..).verify(..)  src/multisig.rs:154-156, 393-429
    pub fn jjs_verify_aggregate(ctx: *mut jjs_ctx, pks32: *const u8, offsets: *const u32, sig64: *const u8,
                                msg32: *const u8, n: usize, status: *mut u8, c32_or_null: *mut u8,
                                aggpk32_or_null: *mut u8) -> c_int;
    // several kinds in one call, balanced over the devices
    pub fn jjs_verify_mixed(ctx: *mut jjs_ctx, parts: *const jjs_part, n_parts: usize) -> c_int;
    // device-buffer entry points (enqueue on the caller's stream)
    pub fn jjs_verify_single_device(ctx: *mut jjs_ctx, device_index: c_int, d_pk32: *const u8, d_sig64: *const u8,
                                    d_msg32: *const u8, n: usize, d_status: *mut u8, d_c32_or_null: *mut u8,
                                    cuda_stream: *mut c_void) -> c_int;
    pub fn jjs_verify_double_device(ctx: *mut jjs_ctx, device_index: c_int, d_pk64: *const u8, d_sig96: *const u8,
                                    d_msg32: *const u8, n: usize, d_status: *mut u8, d_c32_or_null: *mut u8,
                                    cuda_stream: *mut c_void) -> c_int;
    pub fn jjs_verify_vargen_device(ctx: *mut jjs_ctx, device_index: c_int, d_pk64: *const u8, d_sig64: *const u8,
                                    d_msg32: *const u8, n: usize, d_status: *mut u8, d_c32_or_null: *mut u8,
                                    cuda_stream: *mut c_void) -> c_int;
    pub fn jjs_status_bitmap_device(ctx: *mut jjs_ctx, device_index: c_int, d_status: *const u8, n: usize,
                                    d_accept_bitmap: *mut u32, cuda_stream: *mut c_void) -> c_int;
    pub fn jjs_verify_aggregate_device(ctx: *mut jjs_ctx, device_index: c_int, d_pks32: *const u8, d_offsets: *const u32,
                                       h_offsets: *const u32, d_sig64: *const u8, d_msg32: *const u8, n: usize,
                                       d_status: *mut u8, d_c32_or_null: *mut u8, d_aggpk32_or_null: *mut u8,
                                       cuda_stream: *mut c_void) -> c_int;
    // registered key sets (single or double keys): decoded, validated and tabulated once, named by an int handle
    pub fn jjs_keyset_create(ctx: *mut jjs_ctx, kind: c_int, pk: *const u8, n_keys: usize, key_status_or_null: *mut u8,
                             keyset_out: *mut c_int) -> c_int;
    pub fn jjs_keyset_destroy(ctx: *mut jjs_ctx, keyset: c_int) -> c_int;
    pub fn jjs_verify_keyed(ctx: *mut jjs_ctx, keyset: c_int, key_index: *const u32, sig: *const u8, msg32: *const u8, n: usize,
                            status_or_null: *mut u8, c32_or_null: *mut u8, accept_bitmap_or_null: *mut u32) -> c_int;
    pub fn jjs_verify_keyed_device(ctx: *mut jjs_ctx, device_index: c_int, keyset: c_int, d_key_index: *const u32, d_sig: *const u8,
                                   d_msg32: *const u8, n: usize, d_status: *mut u8, d_c32_or_null: *mut u8,
                                   cuda_stream: *mut c_void) -> c_int;
    pub fn jjs_keyset_table_check(ctx: *mut jjs_ctx, keyset: c_int, entries: *const u32, n: usize, mismatches: *mut u32) -> c_int;
    // key sets within a byte budget per device: the widest key-window width 8..4 that fits, else the decoded points only
    pub fn jjs_keyset_create_limited(ctx: *mut jjs_ctx, kind: c_int, pk: *const u8, n_keys: usize, bytes_per_device: usize,
                                     key_status_or_null: *mut u8, keyset_out: *mut c_int) -> c_int;
    pub fn jjs_keyset_info(ctx: *const jjs_ctx, keyset: c_int, key_window_bits: *mut c_int, bytes_per_device: *mut u64) -> c_int;
    // NEW all-or-nothing verification of single / double items by one random linear combination (DESIGN.md section 12)
    pub fn jjs_verify_all(ctx: *mut jjs_ctx, kind: c_int, pk: *const u8, sig: *const u8, msg32: *const u8, n: usize,
                          seed32_or_null: *const u8, all_valid: *mut c_int) -> c_int;
    pub fn jjs_verify_all_device(ctx: *mut jjs_ctx, device_index: c_int, kind: c_int, d_pk: *const u8, d_sig: *const u8,
                                 d_msg32: *const u8, n: usize, seed32_or_null: *const u8, d_all_valid: *mut c_int,
                                 cuda_stream: *mut c_void) -> c_int;
    // NEW all-or-nothing verification of the items of every part, any kind, by one combination (DESIGN.md section 13)
    pub fn jjs_verify_all_mixed(ctx: *mut jjs_ctx, parts: *const jjs_part, n_parts: usize, seed32_or_null: *const u8,
                                all_valid: *mut c_int) -> c_int;
    pub fn jjs_verify_all_mixed_device(ctx: *mut jjs_ctx, device_index: c_int, parts: *const jjs_part, n_parts: usize,
                                       h_offsets_or_null: *const *const u32, seed32_or_null: *const u8, d_all_valid: *mut c_int,
                                       cuda_stream: *mut c_void) -> c_int;
    pub fn jjs_verify_grouped(ctx: *mut jjs_ctx, parts: *const jjs_part, n_parts: usize, seed32_or_null: *const u8,
                              fallback_items_or_null: *mut u64) -> c_int;
    pub fn jjs_verify_grouped_device(ctx: *mut jjs_ctx, device_index: c_int, parts: *const jjs_part, n_parts: usize,
                                     h_offsets_or_null: *const *const u32, seed32_or_null: *const u8,
                                     d_fallback_items_or_null: *mut u64, cuda_stream: *mut c_void) -> c_int;
    // typed inputs: JubJubExtended coordinates, 160 bytes per point (variant 0: PK, R; 1: PK, PK', R, R'; 2: PK, gen, R)
    pub fn jjs_verify_ext(ctx: *mut jjs_ctx, variant: c_int, points_ext160: *const u8, u32_: *const u8, msg32: *const u8,
                          n: usize, status: *mut u8, c32_or_null: *mut u8) -> c_int;
    pub fn jjs_points_to_ext(ctx: *mut jjs_ctx, points32: *const u8, z_mont32: *const u8, n: usize, out160: *mut u8) -> c_int;
    // multisig::combine / verify_share over ragged sessions      src/multisig.rs:255-347, 366-387
    pub fn jjs_multisig_combine(ctx: *mut jjs_ctx, pks32: *const u8, r32: *const u8, s32: *const u8, z32: *const u8,
                                offsets: *const u32, msg32: *const u8, n: usize, share_ok_or_null: *mut u8, status: *mut u8,
                                bad_index_or_null: *mut u32, sig64_or_null: *mut u8) -> c_int;
    pub fn jjs_challenge_only(ctx: *mut jjs_ctx, variant: c_int, pk: *const u8, sig: *const u8, msg32: *const u8, n: usize,
                              c32: *mut u8) -> c_int;
    pub fn jjs_subgroup_check(ctx: *mut jjs_ctx, points32: *const u8, n: usize, method: c_int, out: *mut u8) -> c_int;
    pub fn jjs_fb_table_check(ctx: *mut jjs_ctx, which: c_int, entries: *const u32, n: usize, mismatches: *mut u32) -> c_int;
    pub fn jjs_sign_batch(ctx: *mut jjs_ctx, variant: c_int, sk32: *const u8, rnd32: *const u8, gen_scalar32_or_null: *const u8,
                          msg32: *const u8, n: usize, pk_out: *mut u8, sig_out: *mut u8) -> c_int;
    pub fn jjs_sign_aggregate_batch(ctx: *mut jjs_ctx, sk32: *const u8, offsets: *const u32, rnd32: *const u8, msg32: *const u8,
                                    n: usize, pks32_out: *mut u8, sig64_out: *mut u8) -> c_int;
    pub fn jjs_profile_enable(ctx: *mut jjs_ctx, on: c_int);
    pub fn jjs_profile_collect(ctx: *mut jjs_ctx, stage_ms: *mut f64, stage_count: *mut u64) -> c_int;
    pub fn jjs_launch_count(ctx: *const jjs_ctx) -> u64;
}
