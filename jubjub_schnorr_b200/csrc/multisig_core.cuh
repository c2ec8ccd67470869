// multisig::combine / verify_share for many sessions (SURVEY.md section 8(f) row 2).
//
// Per session (reference src/multisig.rs:311-347, 366-387, 440-500):
//   d_i  = H_trunc(pk_i || pk_1 .. pk_n),  pk_agg = sum d_i pk_i
//   a    = H_trunc(pk_agg || m || R_1 || S_1 || .. || R_n || S_n)
//   RSa  = sum (R_i + a S_i),  c = H_trunc(RSa || pk_agg || m)
//   share i is valid iff  z_i G + (c d_i) pk_i == R_i + a S_i;  the combined signature is (sum z_i, RSa).
// Like the reference, no subgroup validation happens here (the points are only decoded), so the equation is
// evaluated with full-size scalars (the half-size trick of the verify path needs prime-order points).
#pragma once
#include "verify_core.cuh"

namespace jjs {

constexpr uint8_t SF_DECODED = 1;      // every field of the session decodes
constexpr uint8_t SF_NONEMPTY = 2;     // at least one participant (else InvalidMultisigTranscript)

JJS_HD void fr_add(uint32_t* out, const uint32_t* a, const uint32_t* b) {  // a, b < r
    uint32_t s[8], t[8], ord[8];
#pragma unroll
    for (int i = 0; i < 8; i++) ord[i] = JJS_C(R_ORDER)[i];
    add8(s, a, b);
    uint32_t borrow = sub8(t, s, ord);
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = borrow ? s[i] : t[i];
}

// decoded points of the whole batch: index j (pk), K + j (R), 2K + j (S)
JJS_HD void stage_msig_session(const fq* pu, const fq* pv, const uint8_t* pf, size_t K, uint32_t lo, uint32_t hi, const WireField& msg,
                               const WireField& zf, size_t session, uint32_t* d_words, uint32_t* cd_words, uint32_t* a_words, fq* rsa_u, fq* rsa_v,
                               uint8_t* sflags, fq* tabA, size_t stride, const fq* tags) {
    uint32_t w[8];
    fq m;
    wire_load(w, msg, session);
    bool decoded = fq_from_wire(m, w);
    for (uint32_t j = lo; j < hi; j++) {
        decoded = decoded && (pf[j] & PF_DECODED) && (pf[K + j] & PF_DECODED) && (pf[2 * K + j] & PF_DECODED);
        wire_load(w, zf, j);
        decoded = decoded && fr_wire_is_canonical(w);
    }
    uint8_t fl = (decoded ? SF_DECODED : 0) | (hi > lo ? SF_NONEMPTY : 0);
    sflags[session] = fl;
    if (fl != (SF_DECODED | SF_NONEMPTY)) return;
    // aggregate key
    ext acc;
    ext_identity(acc);
#pragma unroll 1
    for (uint32_t j = lo; j < hi; j += AGG_GROUP) aggregate_group(acc, pu, pv, lo, hi, j, j + AGG_GROUP < hi ? j + AGG_GROUP : hi, d_words, tabA, stride, tags);
    fq zi, au, av;
    fq_inv(zi, acc.Z);
    fq_mul(au, acc.X, zi);
    fq_mul(av, acc.Y, zi);
    // a = H(pk_agg, m, R_1, S_1, ..)
    uint32_t a[8];
    {
        Sponge sp;
        sponge_start_tag(sp, tags[3 + 4 * (size_t)(hi - lo)]);
        sponge_absorb(sp, au);
        sponge_absorb(sp, av);
        sponge_absorb(sp, m);
#pragma unroll 1
        for (uint32_t j = lo; j < hi; j++) {
            sponge_absorb(sp, pu[K + j]);
            sponge_absorb(sp, pv[K + j]);
            sponge_absorb(sp, pu[2 * K + j]);
            sponge_absorb(sp, pv[2 * K + j]);
        }
        sponge_squeeze_truncated(a, sp);
    }
    for (int i = 0; i < 8; i++) a_words[8 * session + i] = a[i];
    // RSa = sum R_i + a * sum S_i
    ext sumR, sumS, t;
    ext_identity(sumR);
    ext_identity(sumS);
#pragma unroll 1
    for (uint32_t j = lo; j < hi; j++) {
        ext p;
        pniels np;
        ext_from_affine(p, pu[K + j], pv[K + j]);
        ext_to_pniels(np, p);
        ext_add_pniels<true>(t, sumR, np);
        sumR = t;
        ext_from_affine(p, pu[2 * K + j], pv[2 * K + j]);
        ext_to_pniels(np, p);
        ext_add_pniels<true>(t, sumS, np);
        sumS = t;
    }
    {
        int8_t dA[64];
        recode_signed16(dA, a);
        varbase_table_build_ext(tabA, stride, sumS);
        ext aS;
        varbase_mul<true>(aS, tabA, stride, dA);
        pniels np;
        ext_to_pniels(np, aS);
        ext_add_pniels<true>(t, sumR, np);
    }
    fq ru, rv;
    fq_inv(zi, t.Z);
    fq_mul(ru, t.X, zi);
    fq_mul(rv, t.Y, zi);
    rsa_u[session] = ru;
    rsa_v[session] = rv;
    // c = H(RSa, pk_agg, m), then c * d_i for every participant
    uint32_t c[8];
    {
        Sponge sp;
        sponge_start(sp, 5);
        sponge_absorb(sp, ru);
        sponge_absorb(sp, rv);
        sponge_absorb(sp, au);
        sponge_absorb(sp, av);
        sponge_absorb(sp, m);
        sponge_squeeze_truncated(c, sp);
    }
#pragma unroll 1
    for (uint32_t j = lo; j < hi; j++) {
        uint32_t d[8], cd[8];
        for (int i = 0; i < 8; i++) d[i] = d_words[8 * (size_t)j + i];
        fr_mul(cd, c, d, 500);  // c, d_i < 2^250
        for (int i = 0; i < 8; i++) cd_words[8 * (size_t)j + i] = cd[i];
    }
}

// z_j G + (c d_j) pk_j - a S_j == R_j  (W: window width of fb_g)
template <int W = FB_W>
JJS_HD bool stage_msig_share(const fq* pu, const fq* pv, size_t K, size_t j, const WireField& zf, const uint32_t* cd_words, const uint32_t* a_session,
                             const niels* fb_g, fq* tabA, fq* tabB, size_t stride) {
    uint32_t z[8], cd[8], a[8];
    wire_load(z, zf, j);
    for (int i = 0; i < 8; i++) { cd[i] = cd_words[8 * j + i]; a[i] = a_session[i]; }
    int8_t dA[64], dB[64];
    recode_signed16(dA, cd);
    recode_signed16(dB, a);
    for (int i = 0; i < 64; i++) dB[i] = (int8_t)-dB[i];
    varbase_table_build(tabA, stride, pu[j], pv[j]);
    varbase_table_build(tabB, stride, pu[2 * K + j], pv[2 * K + j]);
    ext acc, zg, sum;
    straus2<64>(acc, tabA, tabB, stride, dA, dB);
    fixedbase_mul<W>(zg, fb_g, z);
    pniels nz;
    ext_to_pniels(nz, zg);
    ext_add_pniels<false>(sum, acc, nz);
    return ext_eq_affine(sum, pu[K + j], pv[K + j]);
}

// status, first failing participant, combined signature
JJS_HD uint8_t stage_msig_finalize(const uint8_t* sflags, const uint8_t* share_ok, uint32_t lo, uint32_t hi, size_t session, const WireField& zf,
                                   const fq* rsa_u, const fq* rsa_v, uint32_t* bad_index, uint32_t* sig16) {
    for (int i = 0; i < 16; i++) sig16[i] = 0;
    *bad_index = 0xffffffffu;
    uint8_t fl = sflags[session];
    if (!(fl & SF_NONEMPTY)) return 4;
    if (!(fl & SF_DECODED)) return 3;
    uint32_t sum[8] = {0, 0, 0, 0, 0, 0, 0, 0}, z[8];
    for (uint32_t j = lo; j < hi; j++) {
        if (!share_ok[j]) {
            *bad_index = j - lo;
            return 5;
        }
        wire_load(z, zf, j);
        fr_add(sum, sum, z);
    }
    for (int i = 0; i < 8; i++) sig16[i] = sum[i];
    point_to_wire(sig16 + 8, rsa_u[session], rsa_v[session]);
    return 0;
}

}  // namespace jjs
