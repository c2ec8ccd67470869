/*
 * jjschnorr_b200 -- C ABI of the B200-native batch verifier for dusk-network/jubjub-schnorr signatures.
 *
 * This is the drop-in boundary for the reference's verify path: every entry point consumes the
 * reference's own wire encodings and reproduces the result of the reference call it replaces, bit for
 * bit.  A Rust caller binds these through `extern "C"` (see INTEGRATION.md); nothing here exposes C++
 * or torch types, nothing throws, and there is no CPU fallback: if no usable CUDA device is present the
 * calls return JJS_ERR_CUDA.
 *
 * Wire encodings (all little-endian, exactly `to_bytes()` of the reference types):
 *   PublicKey        32 B  compressed point                       reference src/keys/public.rs:80-94
 *   Signature        64 B  u (32) || R (32)                       reference src/signatures.rs:101-118
 *   PublicKeyDouble  64 B  pk || pk'                              reference src/keys/public/double.rs:169-186
 *   SignatureDouble  96 B  u || R || R'                           reference src/signatures/double.rs:122-147
 *   PublicKeyVarGen  64 B  pk || generator                        reference src/keys/public/var_gen.rs:54-79
 *   SignatureVarGen  64 B  u || R                                 reference src/signatures/var_gen.rs:95-112
 *   message          32 B  BlsScalar::to_bytes()
 * Arrays are contiguous, item i at base + i * size.
 *
 * Per-item result (status byte), mirroring Result<(), Error> of the reference (src/error.rs:13-26):
 *   JJS_OK                 Ok(())
 *   JJS_INVALID_SIGNATURE  Err(Error::InvalidSignature)   the verification equation does not hold
 *   JJS_INVALID_POINT      Err(Error::InvalidPoint)       a key / signature point fails is_valid()
 *   JJS_BYTES_ERROR        Err(Error::BytesError(_))      some field fails from_bytes()
 * with the reference's precedence: decoding, then point validity, then the equation.
 * The optional challenge output receives c = challenge_hash(..) as JubJubScalar::to_bytes() for items
 * whose status is JJS_OK or JJS_INVALID_SIGNATURE and 32 zero bytes otherwise (the reference does not
 * compute a challenge for those).
 */
#ifndef JJSCHNORR_B200_H
#define JJSCHNORR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JJS_OK 0
#define JJS_INVALID_SIGNATURE 1
#define JJS_INVALID_POINT 2
#define JJS_BYTES_ERROR 3
/* multisig::combine only */
#define JJS_INVALID_MULTISIG_TRANSCRIPT 4
#define JJS_INVALID_MULTISIG_SHARE 5

/* call return codes */
#define JJS_SUCCESS 0
#define JJS_ERR_ARGUMENT (-1)
#define JJS_ERR_CUDA (-2)
#define JJS_ERR_NOMEM (-3)

typedef struct jjs_ctx jjs_ctx;

/* Create a context over the given CUDA device ordinals (n_devices >= 1; devices == NULL means device 0
 * .. n_devices-1).  Builds the per-device constant tables -- among them the fixed-base window tables for the two generators,
 * 2.4 GB each (12 windows of 2^21 points; ~70 ms per device) -- and allocates no batch memory yet; the first verification adds
 * ~9.3 GiB of scratch per device (sized for 2^20 items in flight, whatever the batch size).
 * On failure *out still receives a context, for jjs_last_error only: every other entry point returns JJS_ERR_CUDA on
 * it (there is no CPU fallback) and jjs_destroy frees it. */
int jjs_init(const int* devices, int n_devices, jjs_ctx** out);
/* A context that never holds more than device_memory_limit bytes of device memory on any of its devices: constant tables,
 * fixed-base tables, pipeline scratch, staging, aggregate scratch and registered key sets together.  Everything except key
 * sets is allocated here, so the footprint is known when the call returns.  The library picks the fastest configuration
 * inside the limit: the capacity C (items per pipeline pass) is the largest power of two in [2^12, 2^20] whose scratch
 * (about 4.2 KB per item) fits beside the 12-bit fixed-base tables (21 windows of 2^12 points, 8.3 MB per generator, L2
 * resident); the 21-bit tables of jjs_init (2.4 GB each) are built instead if they fit in what is left.  Every entry point
 * works on such a context and returns the same bytes as on a jjs_init context; batches of any size stream through C items
 * per pass (host-buffer calls in windows of the staging reserved here).  A call that needs more (a larger tag table, more
 * signers in one item than the aggregate key scratch holds, a larger staging window, a key set) grows within the limit or
 * returns JJS_ERR_NOMEM and leaves the context usable.  A multisig session may have at most C participants.
 * JJS_ERR_NOMEM if even the smallest configuration (about 40 MB; the message states it) does not fit, with nothing left
 * allocated and *out an inert context for jjs_last_error, like jjs_init's; JJS_ERR_ARGUMENT for a limit of 0. */
int jjs_init_limited(const int* devices, int n_devices, size_t device_memory_limit, jjs_ctx** out);
/* What the context holds on device device_index: bytes of device memory it allocated, the fixed-base window width of its
 * G / G' tables (21 or 12), and the items per pipeline pass (the largest batch that runs without being cut into passes).
 * A jjs_init context reports width 21, 2^20 items and what it has allocated so far.  Any pointer may be NULL. */
int jjs_memory_info(const jjs_ctx* ctx, int device_index, uint64_t* bytes_held, int* fb_window_bits, uint64_t* items_in_flight);
void jjs_destroy(jjs_ctx* ctx);
/* Human-readable description of the last failure on this context ("" if none). */
const char* jjs_last_error(const jjs_ctx* ctx);
int jjs_device_count(const jjs_ctx* ctx);

/* ---- host-buffer entry points: shard the batch contiguously over the context's devices, copy in,
 *      verify, copy the status bytes (and challenges) back.  All pointers are host memory (pinned or pageable: every
 *      device of the context is driven by its own host thread for the duration of the call, so staged copies from
 *      pageable memory on one device do not hold up the others).  The calls return when everything is done; if a call
 *      fails, the devices are drained first, so nothing still reads or writes the caller's buffers. -------------- */

/* PublicKey::verify for n (key, signature, message) triples.  reference src/keys/public.rs:114-135 */
int jjs_verify_single(jjs_ctx* ctx, const uint8_t* pk32, const uint8_t* sig64, const uint8_t* msg32, size_t n,
                      uint8_t* status, uint8_t* c32_or_null);
/* NEW in this library (BASELINE.json north_star): verify_batch(&[(PublicKey, Signature, BlsScalar)]) -> Vec<bool>.
 * Same work as jjs_verify_single; the result comes back as a packed accept bitmap, bit (i % 32) of word i / 32 set iff
 * PublicKey::verify(pk_i, sig_i, msg_i) is Ok (src/keys/public.rs:114-135).  accept_bitmap has (n + 31) / 32 words;
 * unused high bits of the last word are 0.  The bits are packed on the GPU with one warp ballot per word. */
int jjs_verify_batch(jjs_ctx* ctx, const uint8_t* pk32, const uint8_t* sig64, const uint8_t* msg32, size_t n,
                     uint32_t* accept_bitmap);
/* The same packed accept bitmap for the other three kinds. */
int jjs_verify_batch_double(jjs_ctx* ctx, const uint8_t* pk64, const uint8_t* sig96, const uint8_t* msg32, size_t n,
                            uint32_t* accept_bitmap);
int jjs_verify_batch_vargen(jjs_ctx* ctx, const uint8_t* pk64, const uint8_t* sig64, const uint8_t* msg32, size_t n,
                            uint32_t* accept_bitmap);
int jjs_verify_batch_aggregate(jjs_ctx* ctx, const uint8_t* pks32, const uint32_t* offsets, const uint8_t* sig64,
                               const uint8_t* msg32, size_t n, uint32_t* accept_bitmap);
/* PublicKeyDouble::verify.  reference src/keys/public/double.rs:86-117 */
int jjs_verify_double(jjs_ctx* ctx, const uint8_t* pk64, const uint8_t* sig96, const uint8_t* msg32, size_t n,
                      uint8_t* status, uint8_t* c32_or_null);
/* PublicKeyVarGen::verify.  reference src/keys/public/var_gen.rs:107-133 */
int jjs_verify_vargen(jjs_ctx* ctx, const uint8_t* pk64, const uint8_t* sig64, const uint8_t* msg32, size_t n,
                      uint8_t* status, uint8_t* c32_or_null);
/* multisig::aggregate_pk(&pks[offsets[i]..offsets[i+1]]).verify(sig_i, msg_i).
 * reference src/multisig.rs:154-156, 393-429 then src/keys/public.rs:114-135.
 * offsets has n + 1 entries; aggpk32_or_null receives PublicKey::to_bytes() of each aggregate key.  Any number of signers
 * per item, as in the reference (the sponge tag of a 2 + 2 n element transcript is computed at call time); an item without
 * signers aggregates to the identity and is reported JJS_INVALID_POINT, which is what verify() returns for that key. */
int jjs_verify_aggregate(jjs_ctx* ctx, const uint8_t* pks32, const uint32_t* offsets, const uint8_t* sig64,
                         const uint8_t* msg32, size_t n, uint8_t* status, uint8_t* c32_or_null,
                         uint8_t* aggpk32_or_null);

/* Several batches of different kinds in ONE call (BASELINE.json configs[3] and [4]: var-generator + aggregate-key items,
 * single + double items).  Every part is split evenly over the context's devices (parts below 8 192 items per device go
 * whole to the least loaded device, weighted by the cost of their kind), so each device carries the same share of every
 * kind and all devices finish together; nothing is synchronised between the parts.  Per part, any of status / c32 /
 * aggpk32 / accept_bitmap may be NULL, but status and accept_bitmap not both. */
#define JJS_KIND_SINGLE 0
#define JJS_KIND_DOUBLE 1
#define JJS_KIND_VARGEN 2
#define JJS_KIND_AGGREGATE 3
typedef struct jjs_part {
    int kind;                 /* JJS_KIND_* */
    const uint8_t* pk;        /* kind 0: pk32;  1, 2: pk64;  3: pks32 (ragged, see offsets) */
    const uint32_t* offsets;  /* kind 3: n + 1 entries;  NULL otherwise */
    const uint8_t* sig;       /* kind 1: sig96;  otherwise sig64 */
    const uint8_t* msg32;
    size_t n;
    uint8_t* status;          /* n status bytes */
    uint8_t* c32;             /* n challenges (32 bytes each) */
    uint8_t* aggpk32;         /* kind 3: n aggregate keys */
    uint32_t* accept_bitmap;  /* (n + 31) / 32 words, as jjs_verify_batch */
} jjs_part;
int jjs_verify_mixed(jjs_ctx* ctx, const jjs_part* parts, size_t n_parts);

/* ---- device-buffer entry points: inputs and outputs already live on device `device_index` of the context
 *      (an index into the list given to jjs_init); the work is ordered after everything `cuda_stream` holds at
 *      the call (a cudaStream_t used as is: NULL is the legacy default stream) and is complete when that stream
 *      is: batches above 2^18 items run as sub-chunks on two streams of the context, forked from and joined back
 *      into `cuda_stream` with events.  Calls on one context share its scratch memory, so keep them on one stream
 *      or order them yourself.  No host copies. --- */
int jjs_verify_single_device(jjs_ctx* ctx, int device_index, const uint8_t* d_pk32, const uint8_t* d_sig64,
                             const uint8_t* d_msg32, size_t n, uint8_t* d_status, uint8_t* d_c32_or_null,
                             void* cuda_stream);
int jjs_verify_double_device(jjs_ctx* ctx, int device_index, const uint8_t* d_pk64, const uint8_t* d_sig96,
                             const uint8_t* d_msg32, size_t n, uint8_t* d_status, uint8_t* d_c32_or_null,
                             void* cuda_stream);
int jjs_verify_vargen_device(jjs_ctx* ctx, int device_index, const uint8_t* d_pk64, const uint8_t* d_sig64,
                             const uint8_t* d_msg32, size_t n, uint8_t* d_status, uint8_t* d_c32_or_null,
                             void* cuda_stream);

/* Pack n status bytes (any *_device entry point's output) into the accept bitmap described at jjs_verify_batch;
 * enqueued on `cuda_stream`. */
int jjs_status_bitmap_device(jjs_ctx* ctx, int device_index, const uint8_t* d_status, size_t n, uint32_t* d_accept_bitmap,
                             void* cuda_stream);

/* Aggregate-key verification on device buffers.  d_offsets / h_offsets: the same n + 1 offsets on the device and on
 * the host (the host copy plans the chunks and is only read during the call).  Enqueue-only like the other *_device
 * calls: the ordering of a chunk by signer count happens on the device.  The one exception is growth of the library's
 * key scratch or tag table (the first aggregate call on a device, more than 2^21 signer keys in one 2^18-item chunk, or
 * more than 511 signers in one item), which waits for the device once. */
int jjs_verify_aggregate_device(jjs_ctx* ctx, int device_index, const uint8_t* d_pks32, const uint32_t* d_offsets,
                                const uint32_t* h_offsets, const uint8_t* d_sig64, const uint8_t* d_msg32, size_t n,
                                uint8_t* d_status, uint8_t* d_c32_or_null, uint8_t* d_aggpk32_or_null, void* cuda_stream);

/* ---- registered key sets: many signatures under a stable set of keys (validators, frequent senders, a service's
 *      registered devices).  A key set is decoded and validated once, and with jjs_keyset_create every key point gets a
 *      table of 32 windows x 128 points j 2^(8 w) PK in affine Niels form, 96 B each: 393 216 B per single key, 786 432 B
 *      per double key (pk with G, pk' with G'), on every device of the context.  Verification against it then evaluates
 *      u G + c PK == R from precomputed tables only, and returns exactly what jjs_verify_single (single key sets) or
 *      jjs_verify_double (double key sets) returns for the same items with the keys written out.  jjs_keyset_create_limited
 *      builds narrower tables, or none, within a byte budget.  A key set is named by an int handle owned by the context;
 *      jjs_destroy frees the key sets still registered. --- */

/* Register n_keys >= 1 keys of kind JJS_KIND_SINGLE (pk: n_keys x 32 B, PublicKey) or JJS_KIND_DOUBLE (pk: n_keys x 64 B,
 * PublicKeyDouble) on every device of the context.  Keys that do not decode or fail is_valid() are registered too, so that
 * indices stay dense: items under them get the status verify() gives for those key bytes.  key_status_or_null receives per
 * key 0 (valid), 2 (InvalidPoint) or 3 (BytesError).  Returns JJS_ERR_ARGUMENT for another kind or n_keys == 0 and
 * JJS_ERR_NOMEM, with nothing left allocated, when the tables do not fit.  Synchronous. */
int jjs_keyset_create(jjs_ctx* ctx, int kind, const uint8_t* pk, size_t n_keys, uint8_t* key_status_or_null, int* keyset_out);
/* Free a key set (waits for the devices first).  An unknown or already destroyed handle returns JJS_ERR_ARGUMENT. */
int jjs_keyset_destroy(jjs_ctx* ctx, int keyset);
/* Item i is verified under key key_index[i] of the set, with signature sig (64 B single, 96 B double) and message msg32.
 * An index >= n_keys is reported as a key that does not decode: status JJS_BYTES_ERROR, zero challenge.  Host buffers,
 * sharded over the context's devices like the other host-buffer entry points; status_or_null and accept_bitmap_or_null
 * (layout of jjs_verify_batch) are not both NULL. */
int jjs_verify_keyed(jjs_ctx* ctx, int keyset, const uint32_t* key_index, const uint8_t* sig, const uint8_t* msg32, size_t n,
                     uint8_t* status_or_null, uint8_t* c32_or_null, uint32_t* accept_bitmap_or_null);
/* The same on device buffers of device `device_index`, enqueue-only on cuda_stream like the other device-buffer entry points. */
int jjs_verify_keyed_device(jjs_ctx* ctx, int device_index, int keyset, const uint32_t* d_key_index, const uint8_t* d_sig,
                            const uint8_t* d_msg32, size_t n, uint8_t* d_status, uint8_t* d_c32_or_null, void* cuda_stream);
/* Key-set table self-check (a cross-check hook for the tests, like jjs_fb_table_check): recompute the n entries named by
 * `entries` from their definition j 2^(KW w) PK by plain double-and-add on device 0 and count those that differ, KW being the
 * set's key-window width (jjs_keyset_info).  Flat index (key * points_per_key + point) * E + w * 2^(KW-1) + j - 1, with
 * E = ceil(251 / KW) * 2^(KW-1) entries per key point (4096 at KW = 8: 32 windows x 128), reduced modulo the table size;
 * points_per_key is 1 (single) or 2 (double: pk, then pk').  The table of a key that failed is_valid() is that of the
 * identity.  JJS_ERR_ARGUMENT on a points-only set, which has no table.  Host buffers. */
int jjs_keyset_table_check(jjs_ctx* ctx, int keyset, const uint32_t* entries, size_t n, uint32_t* mismatches);
/* As jjs_keyset_create, holding at most bytes_per_device bytes of device memory per device (and, on a jjs_init_limited
 * context, no more than its limit leaves): the widest key-window width 8..4 that fits, else decoded points only (65 B per key
 * point).  The bound covers the peak of the build, which also holds 32 B of wire key and ceil(251 / KW) x 128 B of window
 * bases per key point until it returns.  Per key point the tables take ceil(251 / KW) x 2^(KW-1) x 96 B: 393 216 B at KW = 8,
 * 221 184 at 7, 129 024 at 6, 78 336 at 5, 48 384 at 4.  A narrower width costs a few additions per equation (12 + 32
 * at 8, 12 + 63 at 4); a points-only set skips decoding the keys and their subgroup tests but evaluates each item's equation as
 * jjs_verify_single does.  Same items, same statuses and challenges as jjs_keyset_create.  JJS_ERR_ARGUMENT for
 * bytes_per_device == 0 and the arguments jjs_keyset_create refuses; JJS_ERR_NOMEM, nothing held, when not even the points
 * fit (the message states what they need).  Synchronous. */
int jjs_keyset_create_limited(jjs_ctx* ctx, int kind, const uint8_t* pk, size_t n_keys, size_t bytes_per_device,
                              uint8_t* key_status_or_null, int* keyset_out);
/* What a key set holds: key-window width (8..4, 0 = points only) and bytes per device (points, flags and tables: what
 * jjs_memory_info's bytes_held grew by on each device, and what jjs_keyset_destroy returns); any pointer may be NULL.
 * JJS_ERR_ARGUMENT for an unknown handle. */
int jjs_keyset_info(const jjs_ctx* ctx, int keyset, int* key_window_bits, uint64_t* bytes_per_device);

/* Typed inputs (what a Rust caller holds before any to_bytes()): every point is given by its JubJubExtended
 * coordinates (u, v, z, t1, t2), each the in-memory BlsScalar of the reference (4 x u64 little-endian Montgomery limbs,
 * R = 2^256): 160 bytes per point.  points_ext160 is item-major, the points of one item in the order
 *   variant 0: PK, R        variant 1: PK, PK', R, R'        variant 2: PK, generator, R
 * u32 = JubJubScalar::to_bytes() of the signature scalar, msg32 = BlsScalar::to_bytes().  The GPU normalises the points
 * (no per-point inversion on the CPU), applies is_valid() exactly as verify() does for typed values -- z != 0, curve
 * equation, t1 t2 consistency, identity, torsion -- and then runs the same pipeline.  Status 3 is returned when u32 / msg32
 * is not canonical or a coordinate is not a reduced field element.  Host buffers. */
int jjs_verify_ext(jjs_ctx* ctx, int variant, const uint8_t* points_ext160, const uint8_t* u32, const uint8_t* msg32,
                   size_t n, uint8_t* status, uint8_t* c32_or_null);

/* Test-data utility for the typed path: wire point i -> the 160-byte coordinates (u z, v z, z, u z, v) with the caller's
 * Montgomery value z (z_mont32, any non-zero reduced field element); zeros if the point does not decode.  Host buffers. */
int jjs_points_to_ext(jjs_ctx* ctx, const uint8_t* points32, const uint8_t* z_mont32, size_t n, uint8_t* out160);

/* multisig::combine for n sessions (reference src/multisig.rs:311-347; the share check is verify_share,
 * src/multisig.rs:255-281, 366-387).  Session i owns participants offsets[i] .. offsets[i+1]-1 of the ragged arrays
 * pks32 (PublicKey::to_bytes), R32 / S32 (compressed commitment points) and z32 (JubJubScalar::to_bytes shares);
 * msg32 has one BlsScalar per session; any number of participants per session.  Per session:
 *   status 0: Ok(Signature), sig64 = (sum z_i) || RSa       5: Err(InvalidMultisigShare(bad_index))
 *          3: some field fails from_bytes                     4: Err(InvalidMultisigTranscript) (no participants)
 * share_ok (one byte per participant) is what verify_share returns for every participant, not only the first bad
 * one.  Like the reference, no subgroup validation is applied to any point.  Host buffers, device 0. */
int jjs_multisig_combine(jjs_ctx* ctx, const uint8_t* pks32, const uint8_t* R32, const uint8_t* S32, const uint8_t* z32,
                         const uint32_t* offsets, const uint8_t* msg32, size_t n, uint8_t* share_ok_or_null, uint8_t* status,
                         uint32_t* bad_index_or_null, uint8_t* sig64_or_null);

/* All-or-nothing verification of n single (kind JJS_KIND_SINGLE: pk32, sig64) or double (JJS_KIND_DOUBLE: pk64, sig96)
 * items.  *all_valid = 1 iff every item would get JJS_OK from jjs_verify_single / jjs_verify_double, except that a batch
 * containing an item whose equation fails is accepted with probability at most 2^-128; an all-valid batch is never
 * rejected.  n == 0 gives 1.  No per-item results: to find the failing items, call jjs_verify_single / _double.
 * One random linear combination of all the equations with secret 128-bit weights, evaluated as a multi-scalar
 * multiplication (DESIGN.md section 12); every point is subgroup-tested.
 * seed32_or_null: NULL draws a fresh 32-byte secret seed from the operating system for every call (what production must
 * do); a caller-given seed makes the call deterministic and is for tests only -- whoever knows the seed can forge a
 * batch that passes.  Other kinds: JJS_ERR_ARGUMENT.  Host buffers, sharded over the context's devices. */
int jjs_verify_all(jjs_ctx* ctx, int kind, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg32, size_t n,
                   const uint8_t* seed32_or_null, int* all_valid);
/* The same on device buffers of device `device_index`; *d_all_valid (device memory, one 32-bit int) is written on cuda_stream,
 * enqueue-only like the other device-buffer entry points; seed32_or_null is host memory, read during the call. */
int jjs_verify_all_device(jjs_ctx* ctx, int device_index, int kind, const uint8_t* d_pk, const uint8_t* d_sig,
                          const uint8_t* d_msg32, size_t n, const uint8_t* seed32_or_null, int* d_all_valid,
                          void* cuda_stream);
/* All-or-nothing verification of every item of every part (jjs_part as for jjs_verify_mixed; any of the four kinds).
 * *all_valid = 1 iff every item would get JJS_OK from jjs_verify_mixed, except that a batch holding an item whose
 * equation fails is accepted with probability at most 2^-128; an all-valid batch is never rejected.  One random linear
 * combination over all parts (DESIGN.md section 13): the weights of an item are those of its position in the whole call
 * (the sizes of the preceding parts plus its index in its part), so a one-part call gives jjs_verify_all's combination for
 * the same seed.  The output fields of every part (status, c32, aggpk32, accept_bitmap) must be NULL.  n_parts == 0 or all
 * parts empty gives 1.  Seed: as jjs_verify_all.  Host buffers, each part sharded over the devices as jjs_verify_mixed
 * shards it.  JJS_ERR_ARGUMENT for an unknown kind, an aggregate part without offsets, a non-NULL output field or a NULL
 * all_valid. */
int jjs_verify_all_mixed(jjs_ctx* ctx, const jjs_part* parts, size_t n_parts, const uint8_t* seed32_or_null, int* all_valid);
/* The same on device buffers of device `device_index`.  The parts' pointers are device memory.  h_offsets_or_null[p] is
 * the host copy of aggregate part p's offsets (the same rule as jjs_verify_aggregate_device), and NULL for other kinds.
 * The whole array may be NULL when no part is aggregate.  Enqueue-only on cuda_stream, with the growth exception of
 * jjs_verify_aggregate_device.  *d_all_valid is device memory. */
int jjs_verify_all_mixed_device(jjs_ctx* ctx, int device_index, const jjs_part* parts, size_t n_parts,
                                const uint32_t* const* h_offsets_or_null, const uint8_t* seed32_or_null,
                                int* d_all_valid, void* cuda_stream);
/* Per-item verification of every item of every part (jjs_part as for jjs_verify_mixed, any of the four kinds, output fields
 * as there: status / c32 / aggpk32 / accept_bitmap, status and accept_bitmap not both NULL).  The outputs are what
 * jjs_verify_mixed writes for the same parts, except that an item whose verification equation fails is reported JJS_OK (and
 * its accept bit set) with probability at most 2^-128.  An item whose equation holds is never misreported, and decoding and
 * point-validity results are exact.  Every item that passes decoding and validity enters a random linear combination of its
 * GROUP: at most 2^16 consecutive items of one pass (DESIGN.md section 14).  Only the items of groups whose combination fails
 * are then verified one by one.  A batch in which few items fail therefore costs about one whole-batch call.  A batch in which
 * most groups hold a failing item costs more than jjs_verify_mixed.
 * *fallback_items_or_null receives the number of items verified one by one (0 for an all-valid batch).
 * Seed: as jjs_verify_all (NULL in production).  Host buffers, parts sharded over the devices as jjs_verify_mixed shards them.
 * JJS_ERR_ARGUMENT for an unknown kind, an aggregate part without offsets, a part with neither status nor accept_bitmap, or
 * NULL parts with n_parts > 0. */
int jjs_verify_grouped(jjs_ctx* ctx, const jjs_part* parts, size_t n_parts, const uint8_t* seed32_or_null,
                       uint64_t* fallback_items_or_null);
/* The same on device buffers of device `device_index`.  Parts and h_offsets_or_null are as for
 * jjs_verify_all_mixed_device, and the output fields of the parts are device memory; here every non-empty part needs its
 * status (accept_bitmap, if given, is computed from it).  *d_fallback_items_or_null (device memory) is written on cuda_stream.
 * The call only enqueues work, with the growth exception of jjs_verify_aggregate_device. */
int jjs_verify_grouped_device(jjs_ctx* ctx, int device_index, const jjs_part* parts, size_t n_parts,
                              const uint32_t* const* h_offsets_or_null, const uint8_t* seed32_or_null,
                              uint64_t* d_fallback_items_or_null, void* cuda_stream);

/* Challenge hash only (hash parity hook): c = challenge_hash(..) for already-valid encodings, no curve
 * check.  variant: 0 single, 1 double, 2 var-generator.  Host buffers. */
int jjs_challenge_only(jjs_ctx* ctx, int variant, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg32,
                       size_t n, uint8_t* c32);

/* is_torsion_free() of n wire-encoded points (reference src/keys/public.rs:160), by the production method
 * (method 0: order-8 Tate pairing) or by the definition (method 1: [r]P == identity by scalar multiplication).
 * out[i] = 1 / 0, or 0xff if the encoding does not decode.  Host buffers; a cross-check hook for the tests. */
int jjs_subgroup_check(jjs_ctx* ctx, const uint8_t* points32, size_t n, int method, uint8_t* out);

/* Fixed-base table self-check (a cross-check hook for the tests, like jjs_subgroup_check): the library builds its window tables
 * for G (which = 0) and G' (which = 1) incrementally; this recomputes the n table entries named by `entries` (flat indices,
 * window * 2^width + digit, reduced modulo the table size) from their definition digit * 2^(width * window) * B by plain
 * double-and-add on device 0 and counts the entries that differ.  Host buffers. */
int jjs_fb_table_check(jjs_ctx* ctx, int which, const uint32_t* entries, size_t n, uint32_t* mismatches);

/* Batch key derivation + signing on device 0 of the context (SURVEY.md section 8(f) row 3; used to make large
 * synthetic batches and by the tests).  For each item: pk = PublicKey::from(&sk) (reference
 * src/keys/public.rs:54-60; PublicKeyDouble / PublicKeyVarGen likewise) and sig = sk.sign(rng, msg) with the
 * reference's hedged nonce (src/keys/secret.rs:174-194, src/nonce.rs:32-86; sign_double: src/keys/secret/double.rs:57-85;
 * var-gen: src/keys/secret/var_gen.rs), where rnd32 is the JubJubScalar the reference draws from its RNG
 * and, for variant 2, the generator is gen_scalar * GENERATOR_EXTENDED as in SecretKeyVarGen::random.
 * All scalars are canonical 32-byte little-endian (sk, rnd, gen_scalar < r; msg < q); an item with an
 * out-of-range input yields all-zero outputs.  Host buffers.  NOT constant-time: test data only. */
int jjs_sign_batch(jjs_ctx* ctx, int variant, const uint8_t* sk32, const uint8_t* rnd32,
                   const uint8_t* gen_scalar32_or_null, const uint8_t* msg32, size_t n, uint8_t* pk_out,
                   uint8_t* sig_out);

/* Synthetic aggregate-key items: signer keys pk_j = sk_j * G (written to pks32_out, ragged like sk32 / offsets, at most 8
 * signers per item), and a hedged Schnorr signature under the aggregate secret sum_j d_j sk_j with the reference's
 * delinearisation coefficients (src/multisig.rs:393-409) -- i.e. what jjs_verify_aggregate accepts.  Host buffers. */
int jjs_sign_aggregate_batch(jjs_ctx* ctx, const uint8_t* sk32, const uint32_t* offsets, const uint8_t* rnd32,
                             const uint8_t* msg32, size_t n, uint8_t* pks32_out, uint8_t* sig64_out);

/* Per-stage device timing (CUDA events on the launching stream around each pipeline stage):
 * stage 0 point decode + subgroup test of the keys, 1 challenge hash, 2 key aggregation (aggregate path only),
 * 3 verification equations, 4 status, 5 deferred subgroup tests of signature points (only those the equation did not
 * already settle).
 * jjs_profile_collect waits for the recorded events, adds their durations (ms) and occurrence counts per
 * stage into the two JJS_N_STAGES-long arrays, and clears the records. */
#define JJS_N_STAGES 6
void jjs_profile_enable(jjs_ctx* ctx, int on);
int jjs_profile_collect(jjs_ctx* ctx, double* stage_ms, uint64_t* stage_count);

/* Kernels launched by this context since creation (for the bench's gpu_launches accounting). */
uint64_t jjs_launch_count(const jjs_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* JJSCHNORR_B200_H */
