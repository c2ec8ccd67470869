// Per-item stages of batch Schnorr verification (single / double / var-generator), shared by the CUDA
// kernels (kernels.cu) and by the CPU twin used in tests/hostsim.
//
// Semantics follow the reference exactly (status codes in include/jjschnorr_b200.h):
//   from_bytes of every field                    -> 3 (BytesError)      reference src/signatures.rs:112-117, src/keys/public.rs:87-94
//   is_valid() of key and signature points       -> 2 (InvalidPoint)    reference src/keys/public.rs:119-121, 159-164
//   c = challenge_hash(..)                                              reference src/signatures.rs:122-141 (+ double.rs:151-177, var_gen.rs:121-142)
//   u*G + c*PK == R (both equations for double)  -> 1 (InvalidSignature) reference src/keys/public.rs:128-132
#pragma once
#include "curve.cuh"
#include "poseidon.cuh"

namespace jjs {

#ifndef JJS_VARGEN_LATTICE
#define JJS_VARGEN_LATTICE 1   // var-generator equation with three short scalars (scalar.cuh, lattice3_reduce); 0: two full-size scalars
#endif

enum Variant : int { VAR_SINGLE = 0, VAR_DOUBLE = 1, VAR_VARGEN = 2 };

// point flags
constexpr uint8_t PF_DECODED = 1;       // from_bytes succeeded
constexpr uint8_t PF_IDENTITY = 2;      // is_identity()
constexpr uint8_t PF_TORSION_FREE = 4;  // is_torsion_free()
constexpr uint8_t PF_TORSION_PENDING = 8;  // subgroup test deferred to the equation stage (signature points, see stage_equation)
// item flags
constexpr uint8_t IF_SCALARS_OK = 1;    // u < r and m < q
constexpr uint8_t IF_EQ0_OK = 2;
constexpr uint8_t IF_EQ1_OK = 4;

struct WireField {
    const uint8_t* base;
    uint32_t stride;
};

JJS_HD void wire_load(uint32_t* w, const WireField& f, size_t i) {
    const uint4* p = reinterpret_cast<const uint4*>(f.base + i * f.stride);
    uint4 a = p[0], b = p[1];
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
    w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
}

// number of point fields per item and their order in the decoded-point arrays
//   single: 0 = PK, 1 = R            double: 0 = PK, 1 = PK', 2 = R, 3 = R'        var-gen: 0 = PK, 1 = generator, 2 = R
JJS_HD int variant_slots(int variant) { return variant == VAR_SINGLE ? 2 : (variant == VAR_DOUBLE ? 4 : 3); }

// ---- stage 1: decode one point ---------------------------------------------------------------
JJS_HD void stage_decode(const WireField& f, size_t item, fq* out_u, fq* out_v, uint8_t* out_flags, size_t slot_index,
                         const Tables& T, bool want_subgroup = true) {
    uint32_t w[8];
    wire_load(w, f, item);
    fq u, v;
    bool ok = point_from_wire(u, v, w, T);
    uint8_t fl = 0;
    if (ok) {
        fq one;
        fq_one(one);
        fl = PF_DECODED | ((fq_is_zero(u) && fq_eq(v, one)) ? PF_IDENTITY : 0);
        if (!want_subgroup) fl |= PF_TORSION_PENDING;
        else if (point_is_torsion_free_tate(u, v)) fl |= PF_TORSION_FREE;
        out_u[slot_index] = u;
        out_v[slot_index] = v;
    }
    out_flags[slot_index] = fl;
}

// ---- stage 1 (typed inputs): one point given as JubJubExtended coordinates (u, v, z, t1, t2) -------------------
// Each coordinate is the in-memory BlsScalar of the reference (4 x u64 little-endian Montgomery limbs, R = 2^256),
// 160 bytes per point.  Mirrors what verify() sees for a typed value (dusk-jubjub semantics, SURVEY A.2):
//   is_on_curve   = z != 0  and  the affine point (u/z, v/z) satisfies the curve equation  and  (u/z)(v/z) z == t1 t2
//   is_identity   = u == 0 and v == z
//   is_torsion_free on the affine point (meaningful only when on the curve; the three are AND-ed by is_valid()).
// A coordinate that is not a reduced field element is reported as undecodable.
JJS_HD void stage_decode_ext(const WireField& f, size_t item, fq* out_u, fq* out_v, uint8_t* out_flags, size_t slot_index,
                             bool want_subgroup = true) {
    fq c[5];
    bool reduced = true;
#pragma unroll
    for (int k = 0; k < 5; k++) {
        WireField fk{f.base + 32 * k, f.stride};
        wire_load(c[k].l, fk, item);
        reduced = reduced && !ge_q(c[k].l);
    }
    if (!reduced) {
        out_flags[slot_index] = 0;
        return;
    }
    fq zi, au, av, u2, v2, lhs, rhs, one, d, t;
    fq_inv(zi, c[2]);
    fq_mul(au, c[0], zi);
    fq_mul(av, c[1], zi);
    fq_sqr(u2, au);
    fq_sqr(v2, av);
    fq_sub(lhs, v2, u2);
    fq_one(one);
    fq_load_const(d, JJS_C(EDWARDS_D));
    fq_mul(rhs, u2, v2);
    fq_mul(rhs, rhs, d);
    fq_add(rhs, rhs, one);
    bool on_curve = !fq_is_zero(c[2]) && fq_eq(lhs, rhs);
    fq_mul(t, au, av);
    fq_mul(t, t, c[2]);
    fq_mul(lhs, c[3], c[4]);
    on_curve = on_curve && fq_eq(t, lhs);
    uint8_t fl = PF_DECODED | ((fq_is_zero(c[0]) && fq_eq(c[1], c[2])) ? PF_IDENTITY : 0);
    // a point off the curve is invalid whatever its subgroup status: its test is neither run nor deferred
    if (on_curve) {
        if (!want_subgroup) fl |= PF_TORSION_PENDING;
        else if (point_is_torsion_free_tate(au, av)) fl |= PF_TORSION_FREE;
    }
    out_u[slot_index] = au;
    out_v[slot_index] = av;
    out_flags[slot_index] = fl;
}

// ---- stage 2: challenge hash -------------------------------------------------------------------
// pts_u / pts_v are [slots][n].  The stage is split the way the kernels run it: (a) scalar range checks and the
// decision whether the item goes on at all, (b) the sponge for the items that do.
JJS_HD bool point_flags_valid(uint8_t f) { return (f & PF_TORSION_FREE) && !(f & PF_IDENTITY); }

// BlsScalar::from_bytes(m) and JubJubScalar::from_bytes(u) succeed (reference src/signatures.rs:113, message decoding)
JJS_HD bool stage_scalars_ok(const WireField& msg, const WireField& usc, size_t item) {
    uint32_t w[8];
    wire_load(w, msg, item);
    bool ok = !ge_q(w);
    wire_load(w, usc, item);
    return ok && fr_wire_is_canonical(w);
}
// An item goes on to the challenge hash and the equations iff every field decoded and -- unless the caller only wants
// challenges -- its keys (and the var-gen generator) are valid: everything else is settled by the flags alone
// (BytesError, or InvalidPoint from a key, both of which the reference reports before it hashes anything).
JJS_HD bool stage_item_ready(int variant, const uint8_t* pflags, size_t n, size_t item, bool scalars_ok, bool require_valid_keys) {
    const int slots = variant_slots(variant), nkeys = variant == VAR_SINGLE ? 1 : 2;
    bool ready = scalars_ok;
    for (int s = 0; s < slots; s++) ready = ready && (pflags[s * n + item] & PF_DECODED);
    if (require_valid_keys)
        for (int s = 0; s < nkeys; s++) ready = ready && point_flags_valid(pflags[s * n + item]);
    return ready;
}
// the sponge of a ready item; writes the challenge as 8 little-endian words
JJS_HD void stage_challenge_hash(int variant, const fq* pts_u, const fq* pts_v, size_t n, size_t item, const WireField& msg, uint32_t* c_out) {
    uint32_t w[8], c[8];
    fq m;
    wire_load(w, msg, item);
    fq_from_wire(m, w);
    Sponge sp;
    if (variant == VAR_SINGLE) {  // [R.u, R.v, pk.u, pk.v, m]
        sponge_start(sp, 5);
        sponge_absorb(sp, pts_u[1 * n + item]);
        sponge_absorb(sp, pts_v[1 * n + item]);
        sponge_absorb(sp, pts_u[0 * n + item]);
        sponge_absorb(sp, pts_v[0 * n + item]);
        sponge_absorb(sp, m);
    } else if (variant == VAR_DOUBLE) {  // [JJSCHDBL, R, R', pk, pk', m]
        sponge_start(sp, 10);
        fq tag;
        fq_load_const(tag, JJS_C(DOUBLE_DOMAIN));
        sponge_absorb(sp, tag);
        sponge_absorb(sp, pts_u[2 * n + item]);
        sponge_absorb(sp, pts_v[2 * n + item]);
        sponge_absorb(sp, pts_u[3 * n + item]);
        sponge_absorb(sp, pts_v[3 * n + item]);
        sponge_absorb(sp, pts_u[0 * n + item]);
        sponge_absorb(sp, pts_v[0 * n + item]);
        sponge_absorb(sp, pts_u[1 * n + item]);
        sponge_absorb(sp, pts_v[1 * n + item]);
        sponge_absorb(sp, m);
    } else {  // [R, pk, generator, m]
        sponge_start(sp, 7);
        sponge_absorb(sp, pts_u[2 * n + item]);
        sponge_absorb(sp, pts_v[2 * n + item]);
        sponge_absorb(sp, pts_u[0 * n + item]);
        sponge_absorb(sp, pts_v[0 * n + item]);
        sponge_absorb(sp, pts_u[1 * n + item]);
        sponge_absorb(sp, pts_v[1 * n + item]);
        sponge_absorb(sp, m);
    }
    sponge_squeeze_truncated(c, sp);
#pragma unroll
    for (int i = 0; i < 8; i++) c_out[item * 8 + i] = c[i];
}
// Both halves for one item (what the work-list kernel and the hash kernel do together).  Returns whether the item is ready;
// the challenge words of an item that is not are zero.
JJS_HD bool stage_challenge(int variant, const fq* pts_u, const fq* pts_v, const uint8_t* pflags, size_t n, size_t item,
                            const WireField& msg, const WireField& usc, uint32_t* c_out, uint8_t* item_flags, bool require_valid_keys = true) {
    bool ok = stage_scalars_ok(msg, usc, item);
    item_flags[item] = ok ? IF_SCALARS_OK : 0;
    bool ready = stage_item_ready(variant, pflags, n, item, ok, require_valid_keys);
    if (ready) stage_challenge_hash(variant, pts_u, pts_v, n, item, msg, c_out);
    else
        for (int i = 0; i < 8; i++) c_out[item * 8 + i] = 0;
    return ready;
}

// ---- subgroup membership of one wire-encoded point, by either method (cross-check hook) ------------
// returns 0xff if the encoding does not decode, else 1 / 0 for is_torsion_free()
JJS_HD uint8_t subgroup_check(const WireField& f, size_t i, int method, fq* tab, size_t stride, const Tables& T) {
    uint32_t w[8];
    wire_load(w, f, i);
    fq u, v;
    if (!point_from_wire(u, v, w, T)) return 0xff;
    if (method == 0) {
        fq one;
        fq_one(one);
        if (fq_is_zero(u) && fq_eq(v, one)) return 1;  // the identity is torsion free by definition
        return point_is_torsion_free_tate(u, v) ? 1 : 0;
    }
    return point_is_torsion_free(tab, stride, u, v) ? 1 : 0;
}

// ---- stage 4: one verification equation  u*B + c*PK == R ------------------------------------------
// Two per-thread tables (tabA, tabB).  Fixed base (base_slot < 0, table `fb`): the challenge is split as
// tau == rho * c (mod r) with ~126-bit tau, rho (half_gcd), and the equivalent check
//     (|rho| u mod r) * B  +  sign(rho) tau * PK  -  |rho| * R  ==  O
// is evaluated with 33 shared-doubling windows instead of 64.  B and PK must lie in the prime-order subgroup (callers
// only evaluate the equation for keys that passed is_valid(), which is also when the reference does).  R need not:
// write R = R0 + T with R0 in the subgroup and T in E[8]; the left side is rho (uB + cPK - R0) - rho T, a subgroup
// part plus a torsion part, and is O only if both vanish.  So
//     check holds and rho odd   =>  T == O (R is torsion free) and u*B + c*PK == R,
//     R torsion free            =>  check holds  <=>  u*B + c*PK == R   (rho is invertible mod r).
// `r_implied` reports the first case: the caller may then take is_torsion_free(R) as established without testing
// it; in every other case it must run the subgroup test on R and use the returned bool only if R passes.
// Variable base (var-gen): three short scalars (below) over 43 windows; the fallback is u*Gen + c*PK by a 64-window Straus
// interleave, compared projectively with R (equality with Gen, PK in the subgroup puts R there too).
// tabA must be followed by two more per-thread tables at tabA + 36 stride (== tabB) and tabA + 72 stride.
// MODE: -1 either kind (decided by base_slot at run time), 0 fixed base only, 1 variable base only -- the kernels instantiate the
// two kinds separately so that neither carries the other's code and registers.  W: window width of the fixed-base table `fb`.
template <int MODE = -1, int W = FB_W>
JJS_HD bool stage_equation(const fq* pts_u, const fq* pts_v, size_t n, size_t item, int pk_slot, int r_slot, int base_slot,
                           const niels* fb, const WireField& usc, const uint32_t* c_words, fq* tabA, fq* tabB, size_t stride,
                           bool* r_implied = nullptr) {
    uint32_t u[8], c[8];
    wire_load(u, usc, item);
#pragma unroll
    for (int i = 0; i < 8; i++) c[i] = c_words[item * 8 + i];
    ext acc;
    if (MODE == 0 || (MODE < 0 && base_slot < 0)) {
        uint32_t tau[5], rho[8];
        bool rho_neg, rho_odd;
        half_gcd(tau, rho, rho_neg, rho_odd, c);
#pragma unroll
        for (int i = 4; i < 8; i++) rho[i] = 0;
        int8_t dT[33], dR[33];
        recode_signed16_33(dT, tau, rho_neg);
        recode_signed16_n<4>(dR, rho, true);
        varbase_table_build(tabA, stride, pts_u[pk_slot * n + item], pts_v[pk_slot * n + item]);
        varbase_table_build(tabB, stride, pts_u[r_slot * n + item], pts_v[r_slot * n + item]);
        straus2<33>(acc, tabA, tabB, stride, dT, dR);
        uint32_t ru[8];
        fr_mul_short(ru, rho, u);  // |rho| * u mod r,  |rho| < 2^126
        fixedbase_acc<W>(acc, fb, ru);
        bool ok = ext_is_identity(acc);
        if (r_implied) *r_implied = ok && rho_odd;
        return ok;
    }
#if JJS_VARGEN_LATTICE
    {
        // three short scalars (scalar.cuh, lattice3_reduce): x*Gen + y*PK - z*R == O over 43 shared-doubling windows and
        // three per-thread tables (tabA, tabB = tabA + 36 stride, and the next one).  The same argument as above covers R:
        // the check passing with z odd proves R torsion free and the equation; otherwise the caller tests R.
        uint32_t xm[8], ym[8], zm[8];
        bool xneg, yneg, zneg, z_odd;
        if (lattice3_reduce(xm, ym, zm, xneg, yneg, zneg, z_odd, u, c)) {
            int8_t dg[3][64];
            recode_signed16_n<6>(dg[0], xm, xneg);
            recode_signed16_n<6>(dg[1], ym, yneg);
            recode_signed16_n<6>(dg[2], zm, !zneg);
            varbase_table_build(tabA, stride, pts_u[base_slot * n + item], pts_v[base_slot * n + item]);
            varbase_table_build(tabA + 36 * stride, stride, pts_u[pk_slot * n + item], pts_v[pk_slot * n + item]);
            varbase_table_build(tabA + 72 * stride, stride, pts_u[r_slot * n + item], pts_v[r_slot * n + item]);
            straus_multi(acc, 3, tabA, stride, dg, LATTICE3_WINDOWS);
            bool ok = ext_is_identity(acc);
            if (r_implied) *r_implied = ok && z_odd;
            return ok;
        }
    }
#endif
    // no short vector found (never seen for hash outputs; reachable in principle): the direct evaluation
    int8_t dU[64], dC[64];
    recode_signed16(dU, u);
    recode_signed16(dC, c);
    varbase_table_build(tabA, stride, pts_u[base_slot * n + item], pts_v[base_slot * n + item]);
    varbase_table_build(tabB, stride, pts_u[pk_slot * n + item], pts_v[pk_slot * n + item]);
    straus2<64>(acc, tabA, tabB, stride, dU, dC);
    bool ok = ext_eq_affine(acc, pts_u[r_slot * n + item], pts_v[r_slot * n + item]);
    if (r_implied) *r_implied = ok;
    return ok;
}

// Equation `eq` of an item, with the deferred subgroup test of its signature point folded in.  Returns the equation
// result and updates the flags of R: PF_TORSION_FREE when the equation implies it; otherwise, if the test is still
// pending, `*need_r_test` is set and the caller must run point_is_torsion_free_tate on R (stage_rtest) before the
// status is formed.  Keys (and the generator) that are not valid make the item InvalidPoint whatever R is, so the
// equation is skipped for them.
JJS_HD void equation_slots(int variant, int eq, int& pk_slot, int& r_slot, int& base_slot) {
    if (variant == VAR_SINGLE) { pk_slot = 0; r_slot = 1; base_slot = -1; }
    else if (variant == VAR_DOUBLE) { pk_slot = eq; r_slot = 2 + eq; base_slot = -1; }
    else { pk_slot = 0; r_slot = 2; base_slot = 1; }
}
template <int MODE = -1, int W = FB_W>
JJS_HD bool stage_equation_item(int variant, int eq, const fq* pts_u, const fq* pts_v, uint8_t* pflags, size_t n, size_t item, const niels* fb,
                                const WireField& usc, const uint32_t* c_words, fq* tabA, fq* tabB, size_t stride, bool* need_r_test) {
    int pk_slot, r_slot, base_slot;
    equation_slots(variant, eq, pk_slot, r_slot, base_slot);
    *need_r_test = false;
    if (!point_flags_valid(pflags[pk_slot * n + item])) return false;
    if (base_slot >= 0 && !point_flags_valid(pflags[base_slot * n + item])) return false;
    bool implied = false;
    bool ok = stage_equation<MODE, W>(pts_u, pts_v, n, item, pk_slot, r_slot, base_slot, fb, usc, c_words, tabA, tabB, stride, &implied);
    uint8_t rf = pflags[r_slot * n + item];
    if (rf & PF_TORSION_PENDING) {
        if (implied) pflags[r_slot * n + item] = (uint8_t)((rf & ~PF_TORSION_PENDING) | PF_TORSION_FREE);
        else *need_r_test = true;
    }
    return ok;
}
// the deferred subgroup test of one decoded point (index into the point arrays)
JJS_HD void stage_rtest(const fq* pts_u, const fq* pts_v, uint8_t* pflags, size_t index) {
    uint8_t f = (uint8_t)(pflags[index] & ~PF_TORSION_PENDING);
    if (point_is_torsion_free_tate(pts_u[index], pts_v[index])) f |= PF_TORSION_FREE;
    pflags[index] = f;
}

// ---- aggregate key: multisig::aggregate_pk (reference src/multisig.rs:154-156, 393-429) ---------------
// keys_u / keys_v / kflags: decoded signer keys of the whole batch (ragged, item i owns [offsets[i], offsets[i+1]));
// d_j = H_trunc(pk_j || pk_0 .. pk_{n-1}),  agg = sum_j d_j * pk_j.  Like the reference, the signer keys are NOT
// validated (only decoded); the aggregate is then treated exactly as the PublicKey of a single verification: its
// affine coordinates, validity flags (identity, torsion freeness) and wire encoding are written to slot `out_index`.
// `tags`: SAFE tags in Montgomery form indexed by the number of absorbed elements (Tables::safe_tags), valid up to 2 + 2 (hi - lo)
JJS_HD void aggregate_coeff_words(uint32_t* d, const fq* keys_u, const fq* keys_v, uint32_t lo, uint32_t hi, uint32_t j, const fq* tags) {
    Sponge sp;
    sponge_start_tag(sp, tags[2 + 2 * (size_t)(hi - lo)]);
    sponge_absorb(sp, keys_u[j]);
    sponge_absorb(sp, keys_v[j]);
#pragma unroll 1
    for (uint32_t k = lo; k < hi; k++) {
        sponge_absorb(sp, keys_u[k]);
        sponge_absorb(sp, keys_v[k]);
    }
    sponge_squeeze_truncated(d, sp);
}

constexpr int AGG_GROUP = 4;  // signer keys folded per shared doubling chain (per-thread tables: AGG_GROUP x R32_TAB_FQ field elements)
constexpr int AGG_DIGITS = 51;  // radix-32 digits of a coefficient below 2^250 (the 51st is at most a carry)

// acc += sum_{j in [j0, j1)} d_j * pk_j,  j1 - j0 <= AGG_GROUP;  optionally stores the coefficients d_j (8 words each)
// `d_ready`: the coefficients were computed by an earlier kernel (stage_aggregate_coeffs) and are read from d_words
JJS_HD void aggregate_group(ext& acc, const fq* keys_u, const fq* keys_v, uint32_t lo, uint32_t hi, uint32_t j0, uint32_t j1, uint32_t* d_words,
                            fq* tab, size_t stride, const fq* tags, bool d_ready = false, bool first_group = false) {
    int8_t digits[AGG_GROUP][R32_DIGITS];
    int nb = 0;
#pragma unroll 1
    for (uint32_t j = j0; j < j1; j++, nb++) {
        uint32_t d[8];
        if (d_ready) {
            for (int i = 0; i < 8; i++) d[i] = d_words[8 * (size_t)j + i];
        } else {
            aggregate_coeff_words(d, keys_u, keys_v, lo, hi, j, tags);
            if (d_words)
                for (int i = 0; i < 8; i++) d_words[8 * (size_t)j + i] = d[i];
        }
        recode_signed32(digits[nb], d);
        varbase_table_build(tab + (size_t)nb * R32_TAB_FQ * stride, stride, keys_u[j], keys_v[j], 16);
    }
    ext term, sum;
    straus_multi32(term, nb, tab, stride, digits, AGG_DIGITS);
    if (first_group) {   // nothing to add it to yet (the usual case: at most AGG_GROUP signers)
        acc = term;
        return;
    }
    pniels nt;
    ext_to_pniels(nt, term);
    ext_add_pniels<true>(sum, acc, nt);
    acc = sum;
}

// whether the signer keys [lo, hi) of an item can be aggregated at all: every key decodes (the reference's from_bytes);
// the number of signers is unbounded, as in the reference
JJS_HD bool aggregate_ready(const uint8_t* kflags, uint32_t lo, uint32_t hi) {
    bool decoded = true;
    for (uint32_t j = lo; j < hi; j++) decoded = decoded && (kflags[j] & PF_DECODED);
    return decoded;
}
// First half of the aggregation as a stage of its own: the delinearisation coefficients d_j of one item (n hashes of
// 2 + 2n elements), written as 8 words each to d_words[8 j ..].  Keeping the hashing apart from the multi-scalar
// multiplication gives two kernels with the register footprint and code size of k_challenge and k_equation.
JJS_HD void stage_aggregate_coeffs(const fq* keys_u, const fq* keys_v, const uint8_t* kflags, uint32_t lo, uint32_t hi, uint32_t* d_words, const fq* tags) {
    if (!aggregate_ready(kflags, lo, hi)) return;
#pragma unroll 1
    for (uint32_t j = lo; j < hi; j++) {
        uint32_t d[8];
        aggregate_coeff_words(d, keys_u, keys_v, lo, hi, j, tags);
#pragma unroll
        for (int i = 0; i < 8; i++) d_words[8 * (size_t)j + i] = d[i];
    }
}
// the same per signer key (what k_agg_coeffs runs: one thread per key, so the hashing of a many-signer item spreads over
// as many threads as it has signers): coefficient of key j of the item owning keys [lo, hi)
JJS_HD void stage_aggregate_coeff_key(const fq* keys_u, const fq* keys_v, const uint8_t* kflags, uint32_t lo, uint32_t hi, uint32_t j, uint32_t* d_words,
                                      const fq* tags) {
    if (!aggregate_ready(kflags, lo, hi)) return;
    uint32_t d[8];
    aggregate_coeff_words(d, keys_u, keys_v, lo, hi, j, tags);
#pragma unroll
    for (int i = 0; i < 8; i++) d_words[8 * (size_t)j + i] = d[i];
}

// The aggregation in two halves around the inversion (sharing one inversion between two items of a thread was measured: no
// gain, the second accumulator spills).  First half: acc = sum_j d_j pk_j in extended coordinates; returns false (acc untouched) if a signer key did not decode.
// d_words: nullptr (coefficients are hashed here) or the output of stage_aggregate_coeffs for the same keys
JJS_HD bool stage_aggregate_point(ext& acc, const fq* keys_u, const fq* keys_v, const uint8_t* kflags, uint32_t lo, uint32_t hi, fq* tab, size_t stride,
                                  const fq* tags, uint32_t* d_words) {
    if (!aggregate_ready(kflags, lo, hi)) return false;
    ext_identity(acc);
#pragma unroll 1
    for (uint32_t j = lo; j < hi; j += AGG_GROUP)
        aggregate_group(acc, keys_u, keys_v, lo, hi, j, j + AGG_GROUP < hi ? j + AGG_GROUP : hi, d_words, tab, stride, tags, d_words != nullptr, j == lo);
    return true;
}
// Second half: affine coordinates from acc and zi = 1 / acc.Z, validity flags, wire encoding (all zero if the keys were not ready)
JJS_HD void stage_aggregate_finish(bool ready, const ext& acc, const fq& zi, fq* out_u, fq* out_v, uint8_t* out_flags, size_t out_index, uint32_t* agg_wire) {
    if (!ready) {
        out_flags[out_index] = 0;
        if (agg_wire)
            for (int i = 0; i < 8; i++) agg_wire[i] = 0;
        return;
    }
    fq u, v, one;
    fq_mul(u, acc.X, zi);
    fq_mul(v, acc.Y, zi);
    fq_one(one);
    uint8_t fl = PF_DECODED | ((fq_is_zero(u) && fq_eq(v, one)) ? PF_IDENTITY : 0);
    if (point_is_torsion_free_tate(u, v)) fl |= PF_TORSION_FREE;
    out_u[out_index] = u;
    out_v[out_index] = v;
    out_flags[out_index] = fl;
    if (agg_wire) point_to_wire(agg_wire, u, v);
}
JJS_HD void stage_aggregate(const fq* keys_u, const fq* keys_v, const uint8_t* kflags, uint32_t lo, uint32_t hi, fq* out_u, fq* out_v,
                            uint8_t* out_flags, size_t out_index, uint32_t* agg_wire, fq* tab, size_t stride, const fq* tags, uint32_t* d_words = nullptr) {
    ext acc;
    bool ready = stage_aggregate_point(acc, keys_u, keys_v, kflags, lo, hi, tab, stride, tags, d_words);
    fq zi;
    if (ready) fq_inv(zi, acc.Z);
    else fq_zero(zi);
    stage_aggregate_finish(ready, acc, zi, out_u, out_v, out_flags, out_index, agg_wire);
}
// ---- stage 5: combine flags into the reference's result -----------------------------------------
JJS_HD uint8_t stage_status(int variant, const uint8_t* pflags, uint8_t item_flags, size_t n, size_t item) {
    const int slots = variant_slots(variant);
    bool decoded = (item_flags & IF_SCALARS_OK) != 0;
    bool valid = true;
    for (int s = 0; s < slots; s++) {
        uint8_t f = pflags[s * n + item];
        decoded = decoded && (f & PF_DECODED);
        valid = valid && (f & PF_TORSION_FREE) && !(f & PF_IDENTITY);
    }
    if (!decoded) return 3;
    if (!valid) return 2;
    bool eq = (item_flags & IF_EQ0_OK) && (variant != VAR_DOUBLE || (item_flags & IF_EQ1_OK));
    return eq ? 0 : 1;
}

}  // namespace jjs
