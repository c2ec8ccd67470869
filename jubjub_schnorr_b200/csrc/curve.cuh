// JubJub (twisted Edwards, a = -1) group arithmetic, point decoding with a table-driven square root, and
// the scalar-multiplication building blocks of the verify path, for sm_100a.
//
// Replaces what the reference reaches through dusk-jubjub: JubJubAffine::from_bytes / from_slice
// (reference src/keys/public.rs:88, src/signatures.rs:114), `point * scalar`, `+`, projective `eq`
// (src/keys/public.rs:128-130), is_torsion_free / is_on_curve / is_identity (src/keys/public.rs:159-164).
#pragma once
#include "consts.cuh"
#include "fq.cuh"
#include "scalar.cuh"

namespace jjs {

JJS_HD void fq_load_const(fq& r, const uint32_t* c) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = c[i];
}

// ---------------------------------------------------------------------------------------------
// large lookup tables living in global memory (device) or in the generated host arrays (hostsim)
// ---------------------------------------------------------------------------------------------
// Fixed-base window width (bits).  One mixed addition per window and no doublings, so wider windows mean fewer additions, and
// HBM is there to be used: 21-bit windows are 12 windows x 2^21 entries x 96 B = 2.4 GB per base (G and G'), one random
// 96-byte read per window.  Measured on B200 per 2^20 single equations: 12 bits (21 windows, 8.3 MB, L2 resident) 26.79 ms,
// 14: 26.48, 16: 26.25, 18: 26.46 (sic), 21 (12 windows): 25.80 -- every window saved is worth its seven products and the DRAM
// reads cost nothing visible next to the ~1 700 products of an equation.  The host twin (tests/hostsim) keeps 12 bits.
#ifndef JJS_FB_W
#if defined(__CUDACC__)
#define JJS_FB_W 21
#else
#define JJS_FB_W 12
#endif
#endif
constexpr int FB_W = JJS_FB_W;
constexpr int FB_WINDOWS = (252 + FB_W - 1) / FB_W;
constexpr int FB_ENTRIES = 1 << FB_W;

struct niels {  // affine Niels form of a fixed-base table entry: (v + u, v - u, 2 d u v)
    fq ypx, ymx, t2d;
};

struct Tables {
    const fq* root_tables;     // [6][256]  g^(-j 2^k) tables for the 2^32-torsion discrete log
    const uint8_t* dlog_hash;  // [1 << JJS_DLOG_HASH_BITS]
    const niels* fb_g;         // [FB_WINDOWS][FB_ENTRIES]  j * 2^(FB_W w) * G
    const niels* fb_gn;        // same for G' (GENERATOR_NUMS_EXTENDED)
    const fq* safe_tags;       // [n]  SAFE sponge tag for n absorbed elements (host-computed, safe_tag.h); multisig transcripts only
};

// ---------------------------------------------------------------------------------------------
// points
// ---------------------------------------------------------------------------------------------
struct ext {  // extended coordinates, u = X/Z, v = Y/Z, T = XY/Z
    fq X, Y, Z, T;
};
struct pniels {  // projective Niels form of a variable-base table entry: (Y + X, Y - X, 2 Z, 2 d T)
    fq ypx, ymx, z2, t2d;
};

JJS_HD void ext_identity(ext& p) {
    fq_zero(p.X);
    fq_one(p.Y);
    fq_one(p.Z);
    fq_zero(p.T);
}
JJS_HD void ext_from_affine(ext& p, const fq& u, const fq& v) {
    p.X = u;
    p.Y = v;
    fq_one(p.Z);
    fq_mul(p.T, u, v);
}
// dbl-2008-hwcd with a = -1: 4S + 4M (3M when the T output is not needed).  With D = -A the formulas
//   E = (X+Y)^2 - A - B, G = D + B, F = G - C, H = D - B,  X3 = E F, Y3 = G H, T3 = E H, Z3 = F G
// are evaluated on the negated quantities E' = A + B - (X+Y)^2, G' = A - B, F' = G' + C, H' = A + B, for which all four
// products keep their sign (E'F' = EF, G'H' = GH, E'H' = EH, F'G' = FG): six additions instead of eight, no negation.
template <bool WANT_T>
JJS_HD void ext_dbl_inl(ext& r, const ext& p) {
    fq a, b, c, e, f, g, h, t;
    fq_sqr(a, p.X);
    fq_sqr(b, p.Y);
    fq_sqr(c, p.Z);
    fq_dbl(c, c);
    fq_add(t, p.X, p.Y);
    fq_sqr(e, t);
    fq_add(h, a, b);   // H'
    fq_sub(e, h, e);   // E'
    fq_sub(g, a, b);   // G'
    fq_add_lazy(f, g, c);   // F' < 2q: its partners in the two products below (E', G') are reduced
    fq_mul(r.X, e, f);
    fq_mul(r.Y, g, h);
    fq_mul(r.Z, f, g);
    if (WANT_T) fq_mul(r.T, e, h);
}
// add-2008-hwcd-3 (a = -1, complete since d is a non-square): extended + projective Niels, 8M (7M without T)
template <bool WANT_T>
JJS_HD void ext_add_pniels_inl(ext& r, const ext& p, const pniels& q) {
    fq a, b, c, d, e, f, g, h, t;
    fq_sub(t, p.Y, p.X);
    fq_mul(a, t, q.ymx);
    fq_add_lazy(t, p.Y, p.X);   // times a reduced table entry
    fq_mul(b, t, q.ypx);
    fq_mul(c, p.T, q.t2d);
    fq_mul(d, p.Z, q.z2);
    fq_sub(e, b, a);
    fq_sub(f, d, c);
    fq_add_lazy(g, d, c);       // its partners (H, F) are reduced
    fq_add(h, b, a);
    fq_mul(r.X, e, f);
    fq_mul(r.Y, g, h);
    fq_mul(r.Z, f, g);
    if (WANT_T) fq_mul(r.T, e, h);
}
// extended + affine Niels (Z2 = 1): 7M (6M without T)
template <bool WANT_T>
JJS_HD void ext_add_niels_inl(ext& r, const ext& p, const niels& q) {
    fq a, b, c, d, e, f, g, h, t;
    fq_sub(t, p.Y, p.X);
    fq_mul(a, t, q.ymx);
    fq_add_lazy(t, p.Y, p.X);   // times a reduced table entry
    fq_mul(b, t, q.ypx);
    fq_mul(c, p.T, q.t2d);
    fq_dbl(d, p.Z);
    fq_sub(e, b, a);
    fq_sub(f, d, c);
    fq_add_lazy(g, d, c);       // its partners (H, F) are reduced
    fq_add(h, b, a);
    fq_mul(r.X, e, f);
    fq_mul(r.Y, g, h);
    fq_mul(r.Z, f, g);
    if (WANT_T) fq_mul(r.T, e, h);
}
// With -DJJS_POINT_CALLS (and -DJJS_INLINE_FIELD) the function-call boundary moves from the field multiplier up to
// the point operations: one call per doubling / addition instead of 7-9 per point operation.
#if defined(__CUDA_ARCH__) && defined(JJS_POINT_CALLS)
template <bool WANT_T>
__device__ __noinline__ ext ext_dbl_fn(ext p) {
    ext r;
    ext_dbl_inl<WANT_T>(r, p);
    if (!WANT_T) r.T = p.T;
    return r;
}
template <bool WANT_T>
__device__ __noinline__ ext ext_add_pniels_fn(ext p, pniels q) {
    ext r;
    ext_add_pniels_inl<WANT_T>(r, p, q);
    if (!WANT_T) r.T = p.T;
    return r;
}
template <bool WANT_T>
__device__ __noinline__ ext ext_add_niels_fn(ext p, niels q) {
    ext r;
    ext_add_niels_inl<WANT_T>(r, p, q);
    if (!WANT_T) r.T = p.T;
    return r;
}
template <bool WANT_T>
JJS_HD void ext_dbl(ext& r, const ext& p) { r = ext_dbl_fn<WANT_T>(p); }
template <bool WANT_T>
JJS_HD void ext_add_pniels(ext& r, const ext& p, const pniels& q) { r = ext_add_pniels_fn<WANT_T>(p, q); }
template <bool WANT_T>
JJS_HD void ext_add_niels(ext& r, const ext& p, const niels& q) { r = ext_add_niels_fn<WANT_T>(p, q); }
#else
template <bool WANT_T>
JJS_HD void ext_dbl(ext& r, const ext& p) { ext_dbl_inl<WANT_T>(r, p); }
template <bool WANT_T>
JJS_HD void ext_add_pniels(ext& r, const ext& p, const pniels& q) { ext_add_pniels_inl<WANT_T>(r, p, q); }
template <bool WANT_T>
JJS_HD void ext_add_niels(ext& r, const ext& p, const niels& q) { ext_add_niels_inl<WANT_T>(r, p, q); }
#endif

JJS_HD void ext_to_pniels(pniels& n, const ext& p) {
    fq d2;
    fq_load_const(d2, JJS_C(EDWARDS_2D));
    fq_add(n.ypx, p.Y, p.X);
    fq_sub(n.ymx, p.Y, p.X);
    fq_dbl(n.z2, p.Z);
    fq_mul(n.t2d, p.T, d2);
}
JJS_HD void pniels_identity(pniels& n) {
    fq_one(n.ypx);
    fq_one(n.ymx);
    fq_one(n.z2);
    fq_dbl(n.z2, n.z2);
    fq_zero(n.t2d);
}
// conditional negation: -(x, y) = (-x, y) swaps ypx/ymx and negates t2d
JJS_HD void pniels_cneg(pniels& n, bool neg) {
    fq nt;
    fq_neg(nt, n.t2d);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint32_t a = n.ypx.l[i], b = n.ymx.l[i];
        n.ypx.l[i] = neg ? b : a;
        n.ymx.l[i] = neg ? a : b;
        n.t2d.l[i] = neg ? nt.l[i] : n.t2d.l[i];
    }
}
JJS_HD bool ext_is_identity(const ext& p) { return fq_is_zero(p.X) && fq_eq(p.Y, p.Z); }
// projective point == affine point (u, v):  X == u Z and Y == v Z   (JubJubExtended::eq with Z2 = 1)
JJS_HD bool ext_eq_affine(const ext& p, const fq& u, const fq& v) {
    fq a, b;
    fq_mul(a, u, p.Z);
    fq_mul(b, v, p.Z);
    return fq_eq(a, p.X) && fq_eq(b, p.Y);
}

// ---------------------------------------------------------------------------------------------
// fixed-exponent powers, inversion, square root of a ratio (q - 1 = 2^32 t)
// ---------------------------------------------------------------------------------------------

// a^e for a fixed exponent given as a generated sliding-window schedule (odd powers a, a^3, ..., a^15):
// entries (squarings, index of the odd power to multiply by, or 0xff for none), most significant window first.
// WHICH = 0: e = (t - 1) / 2 (square root);  WHICH = 1: e = q - 2 (inversion).  The schedules sit in the constant bank.
template <int WHICH>
JJS_HD int pow_sched_entry(int s, int k) { return WHICH == 0 ? JJS_C(SQRT_SCHED)[s][k] : JJS_C(INV_SCHED)[s][k]; }
template <int WHICH>
JJS_HD void fq_pow_sched(fq& r, const fq& a) {
    constexpr int LEN = WHICH == 0 ? JJS_SQRT_SCHED_LEN : JJS_INV_SCHED_LEN;
    fq odd[8], a2;
    odd[0] = a;
    fq_sqr(a2, a);
#pragma unroll 1
    for (int i = 1; i < 8; i++) fq_mul(odd[i], odd[i - 1], a2);
    fq acc = odd[pow_sched_entry<WHICH>(0, 1)];
#pragma unroll 1
    for (int s = 1; s < LEN; s++) {
        int nsq = pow_sched_entry<WHICH>(s, 0), idx = pow_sched_entry<WHICH>(s, 1);
        fq_sqr_n(acc, acc, nsq);
        if (idx != 0xff) fq_mul(acc, acc, odd[idx]);
    }
    r = acc;
}
// a^((t-1)/2)
JJS_HD void fq_pow_tm1d2(fq& r, const fq& a) { fq_pow_sched<0>(r, a); }
// a^(q-2) (Fermat inversion; inv(0) = 0): 254 squarings + 61 products instead of the 164 of square-and-multiply
// On the device the inversion is a real function: it runs once per point or item, and keeping its dynamically
// indexed table of odd powers in a frame of its own avoids the local-array miscompile noted in DESIGN.md section 8
// (seen again when this body was inlined into the key-aggregation kernel).
#if defined(__CUDA_ARCH__)
__device__ __noinline__ fq fq_inv_fn(fq a) {
    fq r;
    fq_pow_sched<1>(r, a);
    return r;
}
JJS_HD void fq_inv(fq& r, const fq& a) { r = fq_inv_fn(a); }
#else
JJS_HD void fq_inv(fq& r, const fq& a) { fq_pow_sched<1>(r, a); }
#endif

JJS_HD uint32_t dlog8(const Tables& T, const fq& x) {  // x in mu_256 = <g^(2^24)>: its discrete log
    uint32_t h = (x.l[0] * JJS_DLOG_HASH_MULT) >> (32 - JJS_DLOG_HASH_BITS);
    return T.dlog_hash[h];
}
JJS_HD void root_table_load(fq& r, const Tables& T, int table, uint32_t j) { r = T.root_tables[table * 256 + j]; }

// r = sqrt(num / den) if it exists (either root); returns false for a non-residue.  den != 0.
// With a = num den, w = a^((t-1)/2), b = a w^2 = a^t lies in the 2^32-torsion <g>; writing b = g^k,
// num / den is a square iff k is even and then sqrt(num/den) = num * w * g^(-k/2).  k is recovered 8 bits
// at a time from b^(2^24), b^(2^16), b^(2^8), b and tables of g^(-j 2^i) (24 squarings + 6 products).
JJS_HD bool fq_sqrt_ratio(fq& r, const fq& num, const fq& den, const Tables& T) {
    fq a, w, b, p1, p2, p3, x, t;
    fq_mul(a, num, den);
    if (fq_is_zero(a)) {
        fq_zero(r);
        return true;
    }
    fq_pow_tm1d2(w, a);
    fq_sqr(b, w);
    fq_mul(b, b, a);
    p1 = b;
    fq_sqr_n(p1, p1, 8);
    p2 = p1;
    fq_sqr_n(p2, p2, 8);
    p3 = p2;
    fq_sqr_n(p3, p3, 8);
    uint32_t k0 = dlog8(T, p3);
    root_table_load(t, T, 2, k0);      // g^(-k0 2^16)
    fq_mul(x, p2, t);
    uint32_t k1 = dlog8(T, x);
    root_table_load(t, T, 1, k0);      // g^(-k0 2^8)
    fq_mul(x, p1, t);
    root_table_load(t, T, 2, k1);      // g^(-k1 2^16)
    fq_mul(x, x, t);
    uint32_t k2 = dlog8(T, x);
    root_table_load(t, T, 0, k0);      // g^(-k0)
    fq_mul(x, b, t);
    root_table_load(t, T, 1, k1);      // g^(-k1 2^8)
    fq_mul(x, x, t);
    root_table_load(t, T, 2, k2);      // g^(-k2 2^16)
    fq_mul(x, x, t);
    uint32_t k3 = dlog8(T, x);
    if (k0 & 1) return false;
    // num * w * g^(-k/2),  k/2 = k0/2 + 2^7 k1 + 2^15 k2 + 2^23 k3
    fq_mul(x, num, w);
    root_table_load(t, T, 0, k0 >> 1);
    fq_mul(x, x, t);
    root_table_load(t, T, 3, k1);
    fq_mul(x, x, t);
    root_table_load(t, T, 4, k2);
    fq_mul(x, x, t);
    root_table_load(t, T, 5, k3);
    fq_mul(r, x, t);
    return true;
}

// ---------------------------------------------------------------------------------------------
// wire decoding
// ---------------------------------------------------------------------------------------------
JJS_HD void load_le32(uint32_t* w, const uint8_t* p) {  // 32 bytes, 4-byte aligned -> 8 little-endian words
    const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = q[i];
}
JJS_HD void store_le32(uint8_t* p, const uint32_t* w) {
    uint32_t* q = reinterpret_cast<uint32_t*>(p);
#pragma unroll
    for (int i = 0; i < 8; i++) q[i] = w[i];
}
// BlsScalar::from_bytes: canonical little-endian, reject >= q.  Output in Montgomery form.
JJS_HD bool fq_from_wire(fq& r, const uint32_t* w) {
    fq raw;
#pragma unroll
    for (int i = 0; i < 8; i++) raw.l[i] = w[i];
    if (ge_q(raw.l)) return false;
    fq_to_mont(r, raw);
    return true;
}
// JubJubScalar::from_bytes: canonical little-endian, reject >= r (reference src/signatures.rs:113)
JJS_HD bool fr_wire_is_canonical(const uint32_t* w) {
    uint32_t ord[8], s[8];
#pragma unroll
    for (int i = 0; i < 8; i++) ord[i] = JJS_C(R_ORDER)[i];
    return sub8(s, w, ord) != 0;  // borrow <=> w < r
}
// JubJubAffine::from_bytes (SURVEY A.3/A.4): v little-endian with the parity of u in bit 255.
// Rejects v >= q, u^2 a non-residue, and u == 0 with the sign bit set.  No subgroup check here.
JJS_HD bool point_from_wire(fq& u, fq& v, const uint32_t* w_in, const Tables& T) {
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = w_in[i];
    uint32_t sign = w[7] >> 31;
    w[7] &= 0x7fffffffu;
    if (!fq_from_wire(v, w)) return false;
    fq v2, num, den, one, d;
    fq_one(one);
    fq_load_const(d, JJS_C(EDWARDS_D));
    fq_sqr(v2, v);
    fq_sub(num, v2, one);
    fq_mul(den, v2, d);
    fq_add(den, den, one);
    if (!fq_sqrt_ratio(u, num, den, T)) return false;
    fq canon;
    fq_from_mont(canon, u);
    bool flip = (canon.l[0] & 1u) != sign;
    fq nu;
    fq_neg(nu, u);
#pragma unroll
    for (int i = 0; i < 8; i++) u.l[i] = flip ? nu.l[i] : u.l[i];
    if (fq_is_zero(u) && sign) return false;
    return true;
}
// JubJubAffine::to_bytes of an affine point given in Montgomery form
JJS_HD void point_to_wire(uint32_t* w, const fq& u, const fq& v) {
    fq cu, cv;
    fq_from_mont(cu, u);
    fq_from_mont(cv, v);
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = cv.l[i];
    w[7] |= (cu.l[0] & 1u) << 31;
}

// ---------------------------------------------------------------------------------------------
// scalar recoding and multiplication
// ---------------------------------------------------------------------------------------------

// signed radix-16 digits d_i in [-8, 8), i = 0..63, of a 256-bit little-endian scalar < 2^253
JJS_HD void recode_signed16(int8_t* digits, const uint32_t* k) {
    uint32_t carry = 0;
#pragma unroll 1
    for (int i = 0; i < 64; i++) {
        int d = (int)((k[i >> 3] >> ((i & 7) * 4)) & 15u) + (int)carry;
        carry = d >= 8;
        digits[i] = (int8_t)(d - (carry << 4));
    }
}

// Per-thread table of 0..8 times a variable base in projective Niels form.  `tab` points at this
// thread's first element; consecutive fq of one entry are `stride` elements apart (device: the batch
// size, so a warp's accesses to one coordinate of one entry are contiguous; host: 1).
JJS_HD void pniels_store(fq* tab, size_t stride, int entry, const pniels& n) {
    fq* p = tab + (size_t)entry * 4 * stride;
    p[0] = n.ypx;
    p[stride] = n.ymx;
    p[2 * stride] = n.z2;
    p[3 * stride] = n.t2d;
}
JJS_HD void pniels_load(pniels& n, const fq* tab, size_t stride, int entry) {
    const fq* p = tab + (size_t)entry * 4 * stride;
    n.ypx = p[0];
    n.ymx = p[stride];
    n.z2 = p[2 * stride];
    n.t2d = p[3 * stride];
}
// entries 0 .. nent of the table: multiples 0, 1, .., nent of p (nent = 8 for radix-16 digits, 16 for radix-32)
JJS_HD void varbase_table_build_ext(fq* tab, size_t stride, const ext& p, int nent = 8) {
    ext acc;
    pniels n1, n;
    pniels_identity(n);
    pniels_store(tab, stride, 0, n);
    ext_to_pniels(n1, p);
    pniels_store(tab, stride, 1, n1);
    acc = p;
#pragma unroll 1
    for (int k = 2; k <= nent; k++) {
        ext_add_pniels<true>(acc, acc, n1);   // in place
        ext_to_pniels(n, acc);
        pniels_store(tab, stride, k, n);
    }
}
JJS_HD void varbase_table_build(fq* tab, size_t stride, const fq& u, const fq& v, int nent = 8) {
    ext p;
    ext_from_affine(p, u, v);
    varbase_table_build_ext(tab, stride, p, nent);
}
// acc = 16 * acc + digit * P, digit in [-8, 8], P's multiples in `tab`
template <bool WANT_T>
JJS_HD void varbase_window(ext& acc, const fq* tab, size_t stride, int digit) {
    ext t;
    ext_dbl<false>(t, acc);
    ext_dbl<false>(acc, t);
    ext_dbl<false>(t, acc);
    ext_dbl<true>(acc, t);
    pniels n;
    int mag = digit < 0 ? -digit : digit;
    pniels_load(n, tab, stride, mag);
    pniels_cneg(n, digit < 0);
    ext_add_pniels<WANT_T>(t, acc, n);
    acc = t;
}
// r = k * P for a table built by varbase_table_build; digits from recode_signed16 (64 digits).
// r.T is only defined when WANT_T.
template <bool WANT_T, typename DIGITS>
JJS_HD void varbase_mul(ext& r, const fq* tab, size_t stride, const DIGITS& digits) {
    ext acc;
    {
        pniels n;
        int d = digits[63];
        int mag = d < 0 ? -d : d;
        pniels_load(n, tab, stride, mag);
        pniels_cneg(n, d < 0);
        ext id;
        ext_identity(id);
        ext_add_pniels<false>(acc, id, n);
    }
#pragma unroll 1
    for (int i = 62; i >= 1; i--) varbase_window<false>(acc, tab, stride, digits[i]);
    varbase_window<WANT_T>(acc, tab, stride, digits[0]);
    r = acc;
}

// acc = 16 acc (T defined on return).  JJS_ROLL_DBL: the three doublings without T as a rolled loop over one inlined copy
// (in place: ext_dbl_inl reads all of its input before it writes), which takes two of the four copies out of the hot loop.
#ifndef JJS_ROLL_DBL
#define JJS_ROLL_DBL 1
#endif
#if JJS_ROLL_DBL
#define JJS_DBL4(acc, t)                                                \
    do {                                                                \
        (void)(t);                                                      \
        _Pragma("unroll 1") for (int k_ = 0; k_ < 3; k_++) ext_dbl<false>(acc, acc); \
        ext_dbl<true>(acc, acc);                                        \
    } while (0)
#else
#define JJS_DBL4(acc, t)          \
    do {                          \
        ext_dbl<false>(t, acc);   \
        ext_dbl<false>(acc, t);   \
        ext_dbl<false>(t, acc);   \
        ext_dbl<true>(acc, t);    \
    } while (0)
#endif

// acc = sum_i 16^i (dA[i] * A + dB[i] * B) over N signed radix-16 digits each (Straus: the doublings are shared);
// tabA / tabB are per-thread tables from varbase_table_build.  acc.T is defined on return.  The second addition of a
// window is followed by a doubling, which does not read T, so it skips that product in every window but the last.
template <int N>
JJS_HD void straus2(ext& r, const fq* tabA, const fq* tabB, size_t stride, const int8_t* dA, const int8_t* dB) {
    ext acc, t;
    pniels n;
    ext_identity(acc);
#pragma unroll 1
    for (int i = N - 1; i >= 0; i--) {
        if (i != N - 1) {
            JJS_DBL4(acc, t);
        }
        int da = dA[i], db = dB[i];
        pniels_load(n, tabA, stride, da < 0 ? -da : da);
        pniels_cneg(n, da < 0);
        ext_add_pniels<true>(t, acc, n);
        pniels_load(n, tabB, stride, db < 0 ? -db : db);
        pniels_cneg(n, db < 0);
        if (i != 0) ext_add_pniels<false>(acc, t, n);
        else ext_add_pniels<true>(acc, t, n);
    }
    r = acc;
}

// acc = sum_b sum_i 16^i d[b][i] * P_b for NB <= 4 variable bases (`nd` <= 64 signed radix-16 digits each) sharing one doubling
// chain; table b lives at tab + b * 36 * stride.  acc.T is defined on return.  The last addition of a window is followed by
// a doubling, which does not read T, so it skips that product in every window but the last.
JJS_HD void straus_multi(ext& r, int nb, const fq* tab, size_t stride, const int8_t (*digits)[64], int nd = 64) {
    ext acc, t;
    pniels n;
    ext_identity(acc);
#pragma unroll 1
    for (int i = nd - 1; i >= 0; i--) {
        if (i != nd - 1) {
            JJS_DBL4(acc, t);
        }
#pragma unroll 1
        for (int b = 0; b < nb; b++) {
            int d = digits[b][i];
            pniels_load(n, tab + (size_t)b * 36 * stride, stride, d < 0 ? -d : d);
            pniels_cneg(n, d < 0);
            // in place: the addition reads all of its first operand before it writes the result
            if (b == nb - 1 && i != 0) ext_add_pniels<false>(acc, acc, n);
            else ext_add_pniels<true>(acc, acc, n);
        }
    }
    r = acc;
}

// ---- radix-32 variant for full-size scalars on several bases (key aggregation) ---------------------------------------------------
// With 250-bit coefficients and up to four bases per doubling chain, 5-bit windows beat 4-bit ones: 51 windows instead of 63
// (13 additions less per base) for eight more table entries per base (72 products): -43 products per base.
constexpr int R32_DIGITS = 52;          // signed radix-32 digits d_i in [-16, 16) of a 256-bit scalar; index 51 is only a carry
constexpr int R32_TAB_FQ = 17 * 4;      // entries 0..16 of a per-thread table, four field elements each
JJS_HD void recode_signed32(int8_t* digits, const uint32_t* k) {
    uint32_t carry = 0;
#pragma unroll 1
    for (int i = 0; i < R32_DIGITS; i++) {
        int bit = 5 * i;
        uint32_t w = 0;
        if (bit < 256) {
            w = k[bit >> 5] >> (bit & 31);
            if ((bit & 31) > 27 && (bit >> 5) + 1 < 8) w |= k[(bit >> 5) + 1] << (32 - (bit & 31));
        }
        int d = (int)(w & 31u) + (int)carry;
        carry = d >= 16;
        digits[i] = (int8_t)(d - (int)(carry << 5));
    }
}
// acc = sum_b sum_i 32^i d[b][i] * P_b for nb <= 4 bases sharing one doubling chain over `nd` radix-32 digits; table b (entries
// 0..16, varbase_table_build with nent = 16) lives at tab + b * R32_TAB_FQ * stride.  acc.T is defined on return.
JJS_HD void straus_multi32(ext& r, int nb, const fq* tab, size_t stride, const int8_t (*digits)[R32_DIGITS], int nd) {
    ext acc;
    pniels n;
    ext_identity(acc);
#pragma unroll 1
    for (int i = nd - 1; i >= 0; i--) {
        if (i != nd - 1) {
#pragma unroll 1
            for (int k = 0; k < 4; k++) ext_dbl<false>(acc, acc);
            ext_dbl<true>(acc, acc);
        }
#pragma unroll 1
        for (int b = 0; b < nb; b++) {
            int d = digits[b][i];
            pniels_load(n, tab + (size_t)b * R32_TAB_FQ * stride, stride, d < 0 ? -d : d);
            pniels_cneg(n, d < 0);
            if (b == nb - 1 && i != 0) ext_add_pniels<false>(acc, acc, n);
            else ext_add_pniels<true>(acc, acc, n);
        }
    }
    r = acc;
}

// Window tables of width W bits: fb_windows(W) windows of 2^W entries.  Every kernel that reads the G / G' tables is instantiated
// at the device default FB_W and at FB_W_SMALL (memory-limited contexts, include/jjschnorr_b200.h jjs_init_limited).
constexpr int FB_W_SMALL = 12;
constexpr int fb_windows(int w) { return (252 + w - 1) / w; }

// r = k * B for a fixed base with precomputed window tables: sum over windows of table[w][k_w] (mixed additions)
template <int W = FB_W>
JJS_HD void fixedbase_mul(ext& r, const niels* table, const uint32_t* k) {
    constexpr int WINDOWS = (252 + W - 1) / W, ENTRIES = 1 << W;
    ext acc;
    ext_identity(acc);
#pragma unroll 1
    for (int w = 0; w < WINDOWS; w++) {
        int bit = w * W;
        uint32_t lo = k[bit >> 5] >> (bit & 31);
        if ((bit & 31) + W > 32 && (bit >> 5) + 1 < 8) lo |= k[(bit >> 5) + 1] << (32 - (bit & 31));
        uint32_t idx = lo & (ENTRIES - 1);
        niels n = table[(size_t)w * ENTRIES + idx];
        ext t;
        ext_add_niels<true>(t, acc, n);
        acc = t;
    }
    r = acc;
}

// acc += k * B (acc.T defined on entry; not on return): the windows are added straight onto a running sum, which saves the
// separate accumulator of fixedbase_mul and the conversion and addition that would join the two
template <int W = FB_W>
JJS_HD void fixedbase_acc(ext& acc, const niels* table, const uint32_t* k) {
    constexpr int WINDOWS = (252 + W - 1) / W, ENTRIES = 1 << W;
#pragma unroll 1
    for (int w = 0; w < WINDOWS; w++) {
        int bit = w * W;
        uint32_t lo = k[bit >> 5] >> (bit & 31);
        if ((bit & 31) + W > 32 && (bit >> 5) + 1 < 8) lo |= k[(bit >> 5) + 1] << (32 - (bit & 31));
        uint32_t idx = lo & (ENTRIES - 1);
        niels n = table[(size_t)w * ENTRIES + idx];
        ext_add_niels<true>(acc, acc, n);   // in place
    }
}

// j * 2^doublings * B in affine coordinates, j < 2^jbits (table construction only)
JJS_HD void fb_affine_multiple(fq& u, fq& v, const fq& bu, const fq& bv, int doublings, int j, int jbits) {
    ext base, acc, t;
    pniels nb;
    ext_from_affine(base, bu, bv);
#pragma unroll 1
    for (int i = 0; i < doublings; i++) {
        ext_dbl<true>(t, base);
        base = t;
    }
    ext_to_pniels(nb, base);
    ext_identity(acc);
#pragma unroll 1
    for (int b = jbits - 1; b >= 0; b--) {
        ext_dbl<true>(t, acc);
        acc = t;
        if ((j >> b) & 1) {
            ext_add_pniels<true>(t, acc, nb);
            acc = t;
        }
    }
    fq zi;
    fq_inv(zi, acc.Z);
    fq_mul(u, acc.X, zi);
    fq_mul(v, acc.Y, zi);
}
JJS_HD void niels_from_affine(niels& out, const fq& u, const fq& v) {
    fq d2;
    fq_load_const(d2, JJS_C(EDWARDS_2D));
    fq_add(out.ypx, v, u);
    fq_sub(out.ymx, v, u);
    fq_mul(out.t2d, u, v);
    fq_mul(out.t2d, out.t2d, d2);
}
// One entry of a fixed-base window table: j * 2^(W w) * B as affine Niels, from scratch (the definition; the device builds
// its tables in two passes, see fb_combine_entries, and the host twin incrementally -- both are checked against this one).
template <int W = FB_W>
JJS_HD void fb_table_entry(niels& out, const fq& bu, const fq& bv, int w, int j) {
    fq u, v;
    fb_affine_multiple(u, v, bu, bv, w * W, j, W);
    niels_from_affine(out, u, v);
}
// Two-pass construction of a window: with j = jh 2^LO + jl the entry is H[jh] + S[jl] for the small tables
// S[jl] = jl 2^(W w) B (2^LO affine points) and H[jh] = jh 2^(W w + LO) B (2^HI points), LO = (W + 1) / 2, HI = W - LO.  A thread combines
// FB_BATCH consecutive entries (same jh) and shares one inversion among them (Montgomery's trick): ~50 products per entry
// instead of the ~1 200 of fb_table_entry, which is what makes 2^21-entry windows cheap to build (12 x 2^21 entries x 2 bases
// in well under a second).
constexpr int FB_BATCH = 8;
JJS_HD void fb_combine_entries(niels* out, const fq* s_u, const fq* s_v, const fq& hu, const fq& hv) {
    ext h, p[FB_BATCH];
    ext_from_affine(h, hu, hv);
    fq prefix[FB_BATCH];
#pragma unroll 1
    for (int k = 0; k < FB_BATCH; k++) {
        niels n;
        niels_from_affine(n, s_u[k], s_v[k]);
        ext_add_niels<false>(p[k], h, n);
        if (k == 0) prefix[0] = p[0].Z;
        else fq_mul(prefix[k], prefix[k - 1], p[k].Z);
    }
    fq inv;
    fq_inv(inv, prefix[FB_BATCH - 1]);   // the addition law is complete: no Z is zero
#pragma unroll 1
    for (int k = FB_BATCH - 1; k >= 0; k--) {
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

// is_torsion_free by the order-8 Tate pairing: E(Fq) is cyclic of order 8 r, so an affine point P != O lies in
// the prime-order subgroup iff tau_8(T8, P) is an 8th power, i.e. g^((q-1)/8) == 1 with
//     g = (N_T V)^4 (N_2T u)^2 (B (1 - v^2))^7,  N_S = B^2 (1+v) - c_S (1-v) u - lam_S B (1+v) u,  V = B (1+v) - x_2T (1-v)
// (derivation and self-test against [r]P on all eight torsion cosets: tools/gen_device_constants.py, tate_constants).
// One fixed exponentiation (~255 squarings) replaces a 252-bit scalar multiplication.  g == 0 exactly for the
// eight torsion points (the identity included: callers flag it separately), all of which are reported "not free".
JJS_HD bool point_is_torsion_free_tate(const fq& u, const fq& v) {
    fq one, opv, omv, t, a, b, nT, n2T, V, h, g, k;
    fq_one(one);
    fq_add(opv, one, v);
    fq_sub(omv, one, v);
    fq_mul(a, omv, u);   // (1-v) u
    fq_mul(b, opv, u);   // (1+v) u
    fq_load_const(k, JJS_C(TATE)[1]);
    fq_mul(t, opv, k);   // B^2 (1+v)
    fq_load_const(k, JJS_C(TATE)[2]);
    fq_mul(nT, a, k);
    fq_sub(nT, t, nT);
    fq_load_const(k, JJS_C(TATE)[3]);
    fq_mul(g, b, k);
    fq_sub(nT, nT, g);
    fq_load_const(k, JJS_C(TATE)[4]);
    fq_mul(n2T, a, k);
    fq_sub(n2T, t, n2T);
    fq_load_const(k, JJS_C(TATE)[5]);
    fq_mul(g, b, k);
    fq_sub(n2T, n2T, g);
    fq_load_const(k, JJS_C(TATE)[0]);
    fq_mul(V, opv, k);   // B (1+v)
    fq_load_const(k, JJS_C(TATE)[6]);
    fq_mul(g, omv, k);
    fq_sub(V, V, g);
    fq_mul(h, opv, omv);  // 1 - v^2
    fq_load_const(k, JJS_C(TATE)[0]);
    fq_mul(h, h, k);
    fq_mul(a, nT, V);
    fq_sqr(a, a);
    fq_sqr(a, a);         // (N_T V)^4
    fq_mul(b, n2T, u);
    fq_sqr(b, b);         // (N_2T u)^2
    fq_mul(g, a, b);
    fq_sqr(a, h);         // h^2
    fq_sqr(b, a);         // h^4
    fq_mul(a, a, h);      // h^3
    fq_mul(a, a, b);      // h^7
    fq_mul(g, g, a);
    // g^((q-1)/8) = (g^t)^(2^29),  g^t = g * (g^((t-1)/2))^2
    fq w;
    fq_pow_tm1d2(w, g);
    fq_sqr(w, w);
    fq_mul(w, w, g);
    fq_sqr_n(w, w, 29);
    return fq_eq(w, one);
}

// [r] P == identity for a point given in affine coordinates (is_torsion_free), by scalar multiplication.
// Kept as the definition-level cross-check of point_is_torsion_free_tate (jjs_subgroup_check, method 1).
JJS_HD bool point_is_torsion_free(fq* tab, size_t stride, const fq& u, const fq& v) {
    varbase_table_build(tab, stride, u, v);
    ext m;
    varbase_mul<false>(m, tab, stride, JJS_C(R_ORDER_DIGITS));
    return ext_is_identity(m);
}

}  // namespace jjs
