// Whole-batch verification by one random linear combination (jjs_verify_all): the building blocks shared by the kernels
// (kernels.cu, run_chunk_rlc) and the CPU twin (tests/hostsim/rlc_twin.cpp).  DESIGN.md section 12.
//
// A batch of n valid-point items is accepted iff
//     (sum z_i u_i) G + sum (z_i c_i) PK_i - sum z_i R_i == O        (double items: the same with z'_i, G', PK'_i, R'_i added)
// A var-generator item contributes (z_i u_i) Gen_i to the multi-scalar multiplication instead of a G term, and an aggregate-key
// item enters as a single item on its aggregate key (DESIGN.md section 13).
// for secret 128-bit weights z_i drawn from a ChaCha20 stream keyed by a 32-byte seed.  The G terms are fixed-base products;
// the rest is one multi-scalar multiplication by buckets (Pippenger): every scalar is cut into signed c-bit digits, each
// digit becomes a (window, bucket) key with a reference to its point, the pairs are radix-sorted by key, the sorted array is
// summed in equal-length segments, and the buckets of each window are weighted by running sums and joined Horner-style.
#pragma once
#include "multisig_core.cuh"   // fr_add

namespace jjs {

// ---- weights: the ChaCha20 block function (RFC 8439 section 2.3) --------------------------------------------------------------
JJS_HD uint32_t rotl32(uint32_t x, int k) { return (x << k) | (x >> (32 - k)); }
JJS_HD void chacha_qr(uint32_t* s, int a, int b, int c, int d) {
    s[a] += s[b]; s[d] = rotl32(s[d] ^ s[a], 16);
    s[c] += s[d]; s[b] = rotl32(s[b] ^ s[c], 12);
    s[a] += s[b]; s[d] = rotl32(s[d] ^ s[a], 8);
    s[c] += s[d]; s[b] = rotl32(s[b] ^ s[c], 7);
}
// out = ChaCha20(key, counter, nonce): sixteen little-endian words (the serialized block of RFC 8439, read as words)
JJS_HD void chacha20_block(uint32_t* out, const uint32_t* key, uint32_t counter, const uint32_t* nonce) {
    uint32_t s[16], x[16];
    s[0] = 0x61707865u; s[1] = 0x3320646eu; s[2] = 0x79622d32u; s[3] = 0x6b206574u;
#pragma unroll
    for (int i = 0; i < 8; i++) s[4 + i] = key[i];
    s[12] = counter;
    s[13] = nonce[0]; s[14] = nonce[1]; s[15] = nonce[2];
#pragma unroll
    for (int i = 0; i < 16; i++) x[i] = s[i];
#pragma unroll 1
    for (int r = 0; r < 10; r++) {
        chacha_qr(x, 0, 4, 8, 12); chacha_qr(x, 1, 5, 9, 13); chacha_qr(x, 2, 6, 10, 14); chacha_qr(x, 3, 7, 11, 15);
        chacha_qr(x, 0, 5, 10, 15); chacha_qr(x, 1, 6, 11, 12); chacha_qr(x, 2, 7, 8, 13); chacha_qr(x, 3, 4, 9, 14);
    }
#pragma unroll
    for (int i = 0; i < 16; i++) out[i] = x[i] + s[i];
}
struct RlcSeed {
    uint32_t w[8];
};
// The weights of the item at position `index` of the whole call: z = words 0..3 and z' = words 4..7 of the block with
// counter = low 32 bits of the index and nonce = (high 32 bits, 0, 0).  A function of the seed and the index only, so the
// weights do not depend on how the call is cut into devices, passes or sub-chunks.
JJS_HD void rlc_weights(uint32_t* z, uint32_t* z2, const RlcSeed& seed, uint64_t index) {
    uint32_t nonce[3] = {(uint32_t)(index >> 32), 0u, 0u}, blk[16];
    chacha20_block(blk, seed.w, (uint32_t)index, nonce);
#pragma unroll
    for (int i = 0; i < 4; i++) { z[i] = blk[i]; z2[i] = blk[4 + i]; }
}

// ---- digits and sort keys -----------------------------------------------------------------------------------------------
// Shape of the combination of one pass: window width c, windows of a full-size scalar (z c mod r < 2^252) and of a weight
// (< 2^128), sort entries per item, the key of an empty entry (zero digit, or an item that is not valid) and the key bits.
// Digits are signed, d in (-2^(c-1), 2^(c-1)]; key = window * 2^(c-1) + |d| - 1, so every key below `sentinel` is a bucket.
// Grouped verification (jjs_verify_grouped, DESIGN.md section 14) cuts a pass into G groups of consecutive items, each with a
// combination of its own: key = (group * nw_big + window) * 2^(c-1) + |d| - 1, so a group's buckets are nw_big more "windows"
// and sorted runs never mix groups.  G = 1 is the whole-batch combination, key for key.
constexpr int RLC_SCALAR_BITS = 252, RLC_WEIGHT_BITS = 128;
constexpr int RLC_C_MIN = 6, RLC_C_MAX = 16;   // at least one 32-bucket slice per window (kernels.cu, RLC_SLICE)
struct RlcShape {
    int c, nw_big, nw_small, per_item;
    uint32_t buckets_per_window, sentinel;
    int end_bit;
};
JJS_HD int rlc_windows(int bits, int c) { return bits / c + 1; }   // the top window absorbs the last carry
// variant: VAR_SINGLE (also aggregate-key items), VAR_DOUBLE or VAR_VARGEN
JJS_HD RlcShape rlc_shape(int variant, int c, size_t groups = 1) {
    RlcShape s;
    s.c = c;
    s.nw_big = rlc_windows(RLC_SCALAR_BITS, c);
    s.nw_small = rlc_windows(RLC_WEIGHT_BITS, c);
    s.per_item = variant == VAR_DOUBLE ? 2 * (s.nw_big + s.nw_small) : (variant == VAR_VARGEN ? 2 * s.nw_big + s.nw_small : s.nw_big + s.nw_small);
    s.buckets_per_window = 1u << (c - 1);
    s.sentinel = (uint32_t)(groups * (size_t)s.nw_big) * s.buckets_per_window;
    s.end_bit = 0;
    while ((1u << s.end_bit) <= s.sentinel) s.end_bit++;
    return s;
}
// bits [pos, pos + c) of an 8-word scalar (zero above bit 255), c <= 16
JJS_HD uint32_t rlc_bits(const uint32_t* k, int pos, int c) {
    if (pos >= 256) return 0;
    const int w = pos >> 5, b = pos & 31;
    uint32_t x = k[w] >> b;
    if (b + c > 32 && w + 1 < 8) x |= k[w + 1] << (32 - b);
    return x & ((1u << c) - 1u);
}
// The entries of one scalar k (nw windows) on point `ref` (index into the point arrays), negated if `neg`: key / value pairs
// keys[w], vals[w] for w < nw; value = ref * 2 + sign.  key0: the first key of the item's group.
JJS_HD void rlc_scalar_entries(uint32_t* keys, uint32_t* vals, const uint32_t* k, int nw, const RlcShape& s, uint32_t ref, bool neg,
                               uint32_t key0 = 0) {
    const uint32_t half = s.buckets_per_window, full = half * 2;
    uint32_t carry = 0;
#pragma unroll 1
    for (int w = 0; w < nw; w++) {
        uint32_t x = rlc_bits(k, w * s.c, s.c) + carry;
        bool dneg = x > half;
        uint32_t mag = dneg ? full - x : x;
        carry = dneg ? 1u : 0u;
        keys[w] = mag ? key0 + (uint32_t)w * half + mag - 1 : s.sentinel;
        vals[w] = ref * 2u + ((dneg != neg) ? 1u : 0u);
    }
}
// Everything one item contributes: weights, z c (and z' c) mod r as the PK scalars, the weights themselves as the (negated)
// R scalars, and z u (z' u) mod r for the G (G') sums.  A var-generator item has no fixed base: z u mod r is a full-size scalar
// on its generator (slot 1) and its G scalar is zero.  `valid`: the item would get status 0 from its equation alone; an item
// that is not valid contributes nothing (sentinel keys, zero G scalars) and the caller clears the batch's validity flag.
// Point references: slot * m + item, the layout of the decoded-point arrays.  Entries: [PK | R | PK' | R'] windows for single
// and double items (aggregate items: the single layout on the aggregate key), [PK | Gen | R] for var-generator items.
// `zu2` is written for double items only.  variant: as rlc_shape.  group: the item's group (0 for a whole-batch pass).
JJS_HD void rlc_item_entries(uint32_t* keys, uint32_t* vals, uint32_t* zu, uint32_t* zu2, int variant, bool valid, const uint32_t* c8,
                             const uint32_t* u8, const RlcSeed& seed, uint64_t index, size_t m, size_t item, const RlcShape& s,
                             uint32_t group = 0) {
    const bool is_double = variant == VAR_DOUBLE;
    if (!valid) {
        for (int e = 0; e < s.per_item; e++) { keys[e] = s.sentinel; vals[e] = 0; }
        for (int i = 0; i < 8; i++) { zu[i] = 0; if (is_double) zu2[i] = 0; }
        return;
    }
    uint32_t z[8] = {0, 0, 0, 0, 0, 0, 0, 0}, z2[8] = {0, 0, 0, 0, 0, 0, 0, 0}, zc[8];
    rlc_weights(z, z2, seed, index);
    const uint32_t key0 = group * (uint32_t)s.nw_big * s.buckets_per_window;
    if (variant == VAR_VARGEN) {
        fr_mul_short(zc, z, c8);
        rlc_scalar_entries(keys, vals, zc, s.nw_big, s, (uint32_t)item, false, key0);
        fr_mul_short(zc, z, u8);
        rlc_scalar_entries(keys + s.nw_big, vals + s.nw_big, zc, s.nw_big, s, (uint32_t)(m + item), false, key0);
        rlc_scalar_entries(keys + 2 * s.nw_big, vals + 2 * s.nw_big, z, s.nw_small, s, (uint32_t)(2 * m + item), true, key0);
        for (int i = 0; i < 8; i++) zu[i] = 0;
        return;
    }
    const int eqs = is_double ? 2 : 1;
    for (int eq = 0; eq < eqs; eq++) {
        const uint32_t* w = eq ? z2 : z;
        const uint32_t pk_ref = (uint32_t)((size_t)eq * m + item), r_ref = (uint32_t)((size_t)(is_double ? 2 + eq : 1) * m + item);
        fr_mul_short(zc, w, c8);
        uint32_t* k = keys + eq * (s.nw_big + s.nw_small);
        uint32_t* v = vals + eq * (s.nw_big + s.nw_small);
        rlc_scalar_entries(k, v, zc, s.nw_big, s, pk_ref, false, key0);
        rlc_scalar_entries(k + s.nw_big, v + s.nw_big, w, s.nw_small, s, r_ref, true, key0);
        fr_mul_short(eq ? zu2 : zu, w, u8);
    }
}

// ---- bucket accumulation over equal-length segments ------------------------------------------------------------------------
// ext + ext (complete)
JJS_HD void rlc_add(ext& acc, const ext& p) {
    pniels n;
    ext_to_pniels(n, p);
    ext t;
    ext_add_pniels<true>(t, acc, n);
    acc = t;
}
// Entry sources of a segment pass: level 0 adds decoded affine points by reference (mixed addition), the merge levels add
// the partial sums of the level below.
struct RlcAffineSrc {
    const fq *u, *v;
    const uint32_t* vals;
    JJS_HD void add(ext& acc, size_t i) const {
        const uint32_t r = vals[i] >> 1;
        niels n;
        niels_from_affine(n, u[r], v[r]);
        if (vals[i] & 1u) {   // -(u, v) = (-u, v)
            fq t = n.ypx;
            n.ypx = n.ymx;
            n.ymx = t;
            fq_neg(n.t2d, n.t2d);
        }
        ext t;
        ext_add_niels<true>(t, acc, n);
        acc = t;
    }
};
struct RlcExtSrc {
    const ext* p;
    JJS_HD void add(ext& acc, size_t i) const { rlc_add(acc, p[i]); }
};
// Segment t = [t L, min((t + 1) L, len)) of a key-sorted array.  Runs of equal keys are summed; a run that neither starts nor
// ends the segment lies wholly inside it and is a finished bucket (written unless it is the sentinel's).  The first and the
// last run of the segment go out as the carries (2t, 2t + 1) -- the last as the identity when the segment holds one run -- so
// the carries are again sorted by key, and the next level sums them the same way.  `final_level` (one segment left): every
// run is finished.  Every thread adds exactly one point per entry, whatever the bucket sizes.  L >= 4, so that every level
// shrinks: s segments leave 2 s carries.
template <typename Src>
JJS_HD void rlc_segment(const uint32_t* keys, const Src& src, size_t len, size_t t, int L, uint32_t sentinel, ext* buckets, uint32_t* ckeys, ext* cpts,
                        bool final_level) {
    const size_t s = t * (size_t)L, e = s + (size_t)L < len ? s + (size_t)L : len;
    if (s >= len) return;
    uint32_t cur = keys[s];
    ext acc;
    ext_identity(acc);
    bool first = true;
#pragma unroll 1
    for (size_t i = s; i < e; i++) {
        const uint32_t k = keys[i];
        if (k != cur) {
            if (first && !final_level) {
                ckeys[2 * t] = cur;
                cpts[2 * t] = acc;
            } else if (cur < sentinel) {
                buckets[cur] = acc;
            }
            first = false;
            cur = k;
            ext_identity(acc);
        }
        if (k < sentinel) src.add(acc, i);
    }
    if (final_level) {
        if (cur < sentinel) buckets[cur] = acc;
        return;
    }
    if (first) {
        ckeys[2 * t] = cur;
        cpts[2 * t] = acc;
        ext_identity(acc);
    }
    ckeys[2 * t + 1] = cur;
    cpts[2 * t + 1] = acc;
}
JJS_HD size_t rlc_segments(size_t len, int L) { return (len + (size_t)L - 1) / (size_t)L; }

// ---- bucket reduction and window combination --------------------------------------------------------------------------------
// r = k p for a small k (double-and-add, most significant bit first)
JJS_HD void rlc_mul_small(ext& r, const ext& p, uint32_t k) {
    ext acc;
    ext_identity(acc);
#pragma unroll 1
    for (int b = 31; b >= 0; b--) {
        ext t;
        ext_dbl<true>(t, acc);
        acc = t;
        if ((k >> b) & 1u) rlc_add(acc, p);
    }
    r = acc;
}
// sum_{j in [lo, hi)} (j + 1) B_j of one window's buckets: running sums from the top give sum (j - lo + 1) B_j, and lo times
// the slice's total supplies the rest
JJS_HD void rlc_bucket_slice(ext& out, const ext* wb, uint32_t lo, uint32_t hi) {
    ext run, sum;
    ext_identity(run);
    ext_identity(sum);
#pragma unroll 1
    for (uint32_t j = hi; j-- > lo;) {
        rlc_add(run, wb[j]);
        rlc_add(sum, run);
    }
    if (lo) {
        ext t;
        rlc_mul_small(t, run, lo);
        rlc_add(sum, t);
    }
    out = sum;
}
// sum_w 2^(c w) W_w, Horner from the top window
JJS_HD void rlc_horner(ext& out, const ext* W, int nw, int c) {
    ext acc = W[nw - 1];
#pragma unroll 1
    for (int w = nw - 2; w >= 0; w--) {
        for (int k = 0; k < c; k++) {
            ext t;
            ext_dbl<true>(t, acc);
            acc = t;
        }
        rlc_add(acc, W[w]);
    }
    out = acc;
}

// The per-scratch-half accumulator of a call: the sum of the passes' MSM results, the G and G' scalar sums mod r, and whether
// every item so far was valid.
struct RlcAcc {
    ext P;
    uint32_t su[2][8];
    uint32_t valid;
};
JJS_HD void rlc_acc_init(RlcAcc& a) {
    ext_identity(a.P);
    for (int i = 0; i < 8; i++) { a.su[0][i] = 0; a.su[1][i] = 0; }
    a.valid = 1;
}
// The G terms, added to the point sum: P + su0 G (+ su1 G' when `with_gn`; a zero su1 adds the identity)
template <int W>
JJS_HD void rlc_fixed_terms(ext& P, const uint32_t (*su)[8], bool with_gn, const niels* fb_g, const niels* fb_gn) {
    ext t;
    fixedbase_mul<W>(t, fb_g, su[0]);
    rlc_add(P, t);
    if (with_gn) {
        fixedbase_mul<W>(t, fb_gn, su[1]);
        rlc_add(P, t);
    }
}

}  // namespace jjs
