// Batch key derivation and signing (SURVEY.md section 8(f) row 3): produces the reference's exact
// PublicKey / Signature bytes from (secret key, RNG scalar, message), so large synthetic batches can be
// made on the GPU instead of on the CPU.  Fixed-base only; not a hot path and not constant-time -- do not
// use it with real secrets.
//
// Mirrors PublicKey::from(&SecretKey) (reference src/keys/public.rs:54-60), SecretKey::sign
// (src/keys/secret.rs:174-194) with hedged_nonce (src/nonce.rs:32-44), SecretKey::sign_double
// (src/keys/secret/double.rs:57-85, nonce tag 2), SecretKeyVarGen::sign (src/keys/secret/var_gen.rs).
#pragma once
#include "verify_core.cuh"

namespace jjs {

JJS_HD void ext_to_affine(fq& u, fq& v, const ext& p) {
    fq zi;
    fq_inv(zi, p.Z);
    fq_mul(u, p.X, zi);
    fq_mul(v, p.Y, zi);
}
// digest_truncated of up to 10 Montgomery inputs
JJS_HD void hash_truncated(uint32_t* c, const fq* in, int n) {
    Sponge sp;
    sponge_start(sp, n);
#pragma unroll 1
    for (int i = 0; i < n; i++) sponge_absorb(sp, in[i]);
    sponge_squeeze_truncated(c, sp);
}
JJS_HD void words_to_fq(fq& r, const uint32_t* w) {  // canonical words (< q) -> Montgomery
    fq raw;
#pragma unroll
    for (int i = 0; i < 8; i++) raw.l[i] = w[i];
    fq_to_mont(r, raw);
}

// variant: 0 single, 1 double, 2 var-generator.  sk, rnd (and gsc for var-gen: generator = gsc * G) are
// JubJub scalars < r as 8 words, msg a BlsScalar < q.  Returns false if an input is out of range.
// Outputs: pk (32 or 64 bytes as words), sig (64 or 96 bytes as words).  W: window width of T's fixed-base tables.
template <int W = FB_W>
JJS_HD bool sign_item(int variant, const uint32_t* sk, const uint32_t* rnd, const uint32_t* gsc, const uint32_t* msg, uint32_t* pk_out,
                      uint32_t* sig_out, const Tables& T) {
    if (!fr_wire_is_canonical(sk) || !fr_wire_is_canonical(rnd) || ge_q(msg)) return false;
    if (variant == VAR_VARGEN && !fr_wire_is_canonical(gsc)) return false;
    fq in[10], m;
    words_to_fq(m, msg);
    uint32_t r[8], c[8], t[8];
    ext P;
    fq gu, gv;
    // hedged nonce
    words_to_fq(in[0], rnd);
    words_to_fq(in[1], sk);
    if (variant == VAR_VARGEN) {
        fixedbase_mul<W>(P, T.fb_g, gsc);
        ext_to_affine(gu, gv, P);
        in[2] = gu; in[3] = gv; in[4] = m;
        hash_truncated(r, in, 5);
    } else {
        uint32_t tag[8] = {variant == VAR_SINGLE ? 1u : 2u, 0, 0, 0, 0, 0, 0, 0};
        words_to_fq(in[2], tag);
        in[3] = m;
        hash_truncated(r, in, 4);
    }
    fq pu, pv, ru, rv, pu2, pv2, ru2, rv2;
    if (variant == VAR_VARGEN) {
        fr_mul(t, sk, gsc);
        fixedbase_mul<W>(P, T.fb_g, t);
        ext_to_affine(pu, pv, P);
        fr_mul(t, r, gsc);
        fixedbase_mul<W>(P, T.fb_g, t);
        ext_to_affine(ru, rv, P);
        in[0] = ru; in[1] = rv; in[2] = pu; in[3] = pv; in[4] = gu; in[5] = gv; in[6] = m;
        hash_truncated(c, in, 7);
        point_to_wire(pk_out, pu, pv);
        point_to_wire(pk_out + 8, gu, gv);
        point_to_wire(sig_out + 8, ru, rv);
    } else {
        fixedbase_mul<W>(P, T.fb_g, sk);
        ext_to_affine(pu, pv, P);
        fixedbase_mul<W>(P, T.fb_g, r);
        ext_to_affine(ru, rv, P);
        point_to_wire(pk_out, pu, pv);
        point_to_wire(sig_out + 8, ru, rv);
        if (variant == VAR_SINGLE) {
            in[0] = ru; in[1] = rv; in[2] = pu; in[3] = pv; in[4] = m;
            hash_truncated(c, in, 5);
        } else {
            fixedbase_mul<W>(P, T.fb_gn, sk);
            ext_to_affine(pu2, pv2, P);
            fixedbase_mul<W>(P, T.fb_gn, r);
            ext_to_affine(ru2, rv2, P);
            point_to_wire(pk_out + 8, pu2, pv2);
            point_to_wire(sig_out + 16, ru2, rv2);
            fq_load_const(in[0], JJS_C(DOUBLE_DOMAIN));
            in[1] = ru; in[2] = rv; in[3] = ru2; in[4] = rv2; in[5] = pu; in[6] = pv; in[7] = pu2; in[8] = pv2; in[9] = m;
            hash_truncated(c, in, 10);
        }
    }
    // u = r - c * sk
    fr_mul(t, c, sk);
    fr_sub(sig_out, r, t);
    return true;
}

}  // namespace jjs
