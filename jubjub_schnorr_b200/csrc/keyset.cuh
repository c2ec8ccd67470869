// Registered key sets: verification against keys that were decoded, validated and tabulated once, ahead of the batch.
// Shared by the CUDA kernels (kernels.cu) and by the CPU twin in tests/hostsim.
//
// With the key known in advance, c * PK is a fixed-base product like u * G: every key point gets a table of signed
// radix-2^KW windows, entry (w, j) = j 2^(KW w) PK for j = 1 .. 2^(KW - 1), in affine Niels form.  The equation
// u*G + c*PK == R is then 12 + keyed_windows(KW) mixed additions (44 at KW = 8) and one projective comparison with R: no
// doublings, no half-gcd and no per-thread table.  Equality also settles R's subgroup membership: G and PK lie in the
// prime-order subgroup, so an R equal to u*G + c*PK lies there too (the argument of the var-generator fallback).  An equation
// that fails leaves R to the deferred subgroup test, and the status is formed from the flags exactly as for unregistered keys.
//
// The key-window width KW is a template parameter of the helpers below, KEYED_MIN_W .. KEYED_MAX_W: narrower windows cost a
// few additions per equation and shrink the table (393 216 B per key point at 8 bits, 48 384 B at 4).  jjs_keyset_create
// builds KEYED_W = 8; jjs_keyset_create_limited takes the widest width whose tables fit the caller's budget.
#pragma once
#include <type_traits>

#include "verify_core.cuh"

namespace jjs {

#ifndef JJS_KEYED_W
#define JJS_KEYED_W 8
#endif
constexpr int KEYED_MIN_W = 4, KEYED_MAX_W = 8;
constexpr int KEYED_W = JJS_KEYED_W;   // the width jjs_keyset_create builds
static_assert(KEYED_W >= KEYED_MIN_W && KEYED_W <= KEYED_MAX_W, "key-table window width");
// challenges are below 2^250: with signed digits in (-2^(KW-1), 2^(KW-1)] the last window absorbs the final carry when KW windows
// cover 251 bits
JJS_HD constexpr int keyed_windows(int kw) { return (251 + kw - 1) / kw; }
JJS_HD constexpr int keyed_entries(int kw) { return 1 << (kw - 1); }                         // j = 1 .. keyed_entries per window
JJS_HD constexpr int keyed_point_entries(int kw) { return keyed_windows(kw) * keyed_entries(kw); }  // per key point: 4 096 at KW = 8
// the geometry of jjs_keyset_create's tables (KW = KEYED_W)
constexpr int KEYED_WINDOWS = keyed_windows(KEYED_W);
constexpr int KEYED_ENTRIES = keyed_entries(KEYED_W);
constexpr int KEYED_POINT_ENTRIES = keyed_point_entries(KEYED_W);  // 4 096 x 96 B = 384 KiB for KW = 8
constexpr int KEYED_BATCH = 8;                                     // entries built per thread around one shared inversion
static_assert(keyed_entries(KEYED_MIN_W) % KEYED_BATCH == 0, "a window splits into whole batches at every width");

// f(std::integral_constant<int, KW>{}) for a run-time key-window width kw in KEYED_MIN_W .. KEYED_MAX_W: the one dispatch from a
// key set's width to the template instances (host code: the library's launches and the CPU twin)
template <typename F>
auto with_key_width(int kw, F&& f) {
    static_assert(KEYED_MIN_W == 4 && KEYED_MAX_W == 8, "one case per width");
    switch (kw) {
    case 8: return f(std::integral_constant<int, 8>{});
    case 7: return f(std::integral_constant<int, 7>{});
    case 6: return f(std::integral_constant<int, 6>{});
    case 5: return f(std::integral_constant<int, 5>{});
    default: return f(std::integral_constant<int, 4>{});
    }
}

// Key points per registered key: single keys have PK, double keys PK (with G) and PK' (with G').
JJS_HD int keyed_points(int variant) { return variant == VAR_DOUBLE ? 2 : 1; }

// The point a key point's table is built for: the key itself when it passed is_valid(), else the identity.  Items under an
// invalid key never reach the equation; the substitution keeps the table (and its check) well defined.
JJS_HD void keyed_table_base(fq& u, fq& v, const fq& ku, const fq& kv, uint8_t kflags) {
    if (point_flags_valid(kflags)) {
        u = ku;
        v = kv;
    } else {
        fq_zero(u);
        fq_one(v);
    }
}

// Table construction, pass 1: bases[w * stride] = 2^(KW w) * (u, v), extended coordinates, for every window.
template <int KW = KEYED_W>
JJS_HD void keyed_window_bases(ext* bases, size_t stride, const fq& u, const fq& v) {
    ext p;
    ext_from_affine(p, u, v);
#pragma unroll 1
    for (int w = 0; w < keyed_windows(KW); w++) {
        bases[(size_t)w * stride] = p;
        if (w + 1 < keyed_windows(KW))
#pragma unroll 1
            for (int k = 0; k < KW; k++) ext_dbl<true>(p, p);
    }
}

// Pass 2: entries j0 .. j0 + KEYED_BATCH - 1 (j0 >= 1) of the window whose base is `base`: j0 * base by double-and-add, the
// rest by repeated addition, all in extended coordinates, then one inversion for the batch (Montgomery's trick, as
// fb_combine_entries).  out[k] is entry j0 + k.
template <int KW = KEYED_W>
JJS_HD void keyed_combine_entries(niels* out, const ext& base, int j0) {
    pniels nb;
    ext_to_pniels(nb, base);
    ext p[KEYED_BATCH];
    ext_identity(p[0]);
#pragma unroll 1
    for (int b = KW - 1; b >= 0; b--) {
        ext_dbl<true>(p[0], p[0]);
        if ((j0 >> b) & 1) ext_add_pniels<true>(p[0], p[0], nb);
    }
    fq prefix[KEYED_BATCH];
    prefix[0] = p[0].Z;
#pragma unroll 1
    for (int k = 1; k < KEYED_BATCH; k++) {
        ext_add_pniels<true>(p[k], p[k - 1], nb);
        fq_mul(prefix[k], prefix[k - 1], p[k].Z);
    }
    fq inv;
    fq_inv(inv, prefix[KEYED_BATCH - 1]);   // the addition law is complete: no Z is zero
#pragma unroll 1
    for (int k = KEYED_BATCH - 1; k >= 0; k--) {
        fq zi, u, v;
        if (k == 0) zi = inv;
        else {
            fq_mul(zi, inv, prefix[k - 1]);
            fq_mul(inv, inv, p[k].Z);
        }
        fq_mul(u, p[k].X, zi);
        fq_mul(v, p[k].Y, zi);
        niels_from_affine(out[k], u, v);
    }
}

// One table entry from its definition, j * 2^(KW w) * B by plain double-and-add (jjs_keyset_table_check and the twin's
// tests compare the built tables with it).
template <int KW = KEYED_W>
JJS_HD void keyed_table_entry(niels& out, const fq& bu, const fq& bv, int w, int j) {
    fq u, v;
    fb_affine_multiple(u, v, bu, bv, w * KW, j, KW);
    niels_from_affine(out, u, v);
}

// acc += c * PK from the key point's table (keyed_point_entries(KW) entries, window-major), c < 2^250; acc.T defined on entry
// and on return.  Digit d of window w selects entry |d| - 1, negated for d < 0 (swap v + u and v - u, negate 2duv); a zero
// digit adds the identity (1, 1, 0) through a select, so every lane runs the same additions.
template <int KW = KEYED_W>
JJS_HD void keyed_acc(ext& acc, const niels* tab, const uint32_t* c) {
    int carry = 0;
#pragma unroll 1
    for (int w = 0; w < keyed_windows(KW); w++) {
        const int bit = w * KW;
        uint32_t raw = bit < 256 ? c[bit >> 5] >> (bit & 31) : 0u;
        if (bit < 256 && (bit & 31) + KW > 32 && (bit >> 5) + 1 < 8) raw |= c[(bit >> 5) + 1] << (32 - (bit & 31));
        int d = (int)(raw & ((2u << (KW - 1)) - 1u)) + carry;
        carry = d > keyed_entries(KW);
        d -= carry << KW;
        const int mag = d < 0 ? -d : d;
        niels n = tab[(size_t)w * keyed_entries(KW) + (mag ? mag - 1 : 0)];
        fq nt, one;
        fq_neg(nt, n.t2d);
        fq_one(one);
        const bool neg = d < 0, zero = mag == 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            uint32_t a = n.ypx.l[i], b = n.ymx.l[i];
            n.ypx.l[i] = zero ? one.l[i] : (neg ? b : a);
            n.ymx.l[i] = zero ? one.l[i] : (neg ? a : b);
            n.t2d.l[i] = zero ? 0u : (neg ? nt.l[i] : n.t2d.l[i]);
        }
        ext_add_niels<true>(acc, acc, n);   // in place
    }
}

// ---- per-item stages ---------------------------------------------------------------------------------------------
// Key slots of item `item` (slot s of the n-item point arrays) from the key set: n_keys keys, their points slot-major
// (key point s of key k at s * n_keys + k).  An index out of range leaves the slots undecoded (BytesError, as a key
// that does not decode).
JJS_HD void stage_keyed_gather(int variant, const fq* keys_u, const fq* keys_v, const uint8_t* kflags, size_t n_keys, uint32_t key,
                               fq* pts_u, fq* pts_v, uint8_t* pflags, size_t n, size_t item) {
    const int nk = keyed_points(variant);
    for (int s = 0; s < nk; s++) {
        uint8_t f = 0;
        if (key < n_keys) {
            const size_t k = (size_t)s * n_keys + key;
            f = kflags[k];
            pts_u[(size_t)s * n + item] = keys_u[k];
            pts_v[(size_t)s * n + item] = keys_v[k];
        }
        pflags[(size_t)s * n + item] = f;
    }
}

// Equation `eq` of an item under a registered key: u*B + c*PK == R with both products from tables (`fb` for B = G or G',
// `ktab` the key point's table).  Updates R's flags like stage_equation_item: PF_TORSION_FREE when the equation holds,
// otherwise `*need_r_test` if R's subgroup test is still pending.  W: window width of `fb`; KW: that of `ktab`.
template <int W = FB_W, int KW = KEYED_W>
JJS_HD bool stage_equation_keyed(int variant, int eq, const fq* pts_u, const fq* pts_v, uint8_t* pflags, size_t n, size_t item, const niels* fb,
                                 const niels* ktab, const WireField& usc, const uint32_t* c_words, bool* need_r_test) {
    int pk_slot, r_slot, base_slot;
    equation_slots(variant, eq, pk_slot, r_slot, base_slot);
    *need_r_test = false;
    if (!point_flags_valid(pflags[pk_slot * n + item])) return false;
    uint32_t u[8], c[8];
    wire_load(u, usc, item);
#pragma unroll
    for (int i = 0; i < 8; i++) c[i] = c_words[item * 8 + i];
    ext acc;
    ext_identity(acc);
    keyed_acc<KW>(acc, ktab, c);
    fixedbase_acc<W>(acc, fb, u);
    const bool ok = ext_eq_affine(acc, pts_u[r_slot * n + item], pts_v[r_slot * n + item]);
    uint8_t rf = pflags[r_slot * n + item];
    if (rf & PF_TORSION_PENDING) {
        if (ok) pflags[r_slot * n + item] = (uint8_t)((rf & ~PF_TORSION_PENDING) | PF_TORSION_FREE);
        else *need_r_test = true;
    }
    return ok;
}

// Status of one registered key (0 valid, 2 InvalidPoint, 3 BytesError): what verify() reports for an otherwise valid item under it.
JJS_HD uint8_t keyed_key_status(int variant, const uint8_t* kflags, size_t n_keys, size_t key) {
    bool decoded = true, valid = true;
    for (int s = 0; s < keyed_points(variant); s++) {
        uint8_t f = kflags[(size_t)s * n_keys + key];
        decoded = decoded && (f & PF_DECODED);
        valid = valid && point_flags_valid(f);
    }
    return !decoded ? 3 : (!valid ? 2 : 0);
}

}  // namespace jjs
