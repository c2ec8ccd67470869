// CPU twin of whole-batch verification (csrc/rlc.cuh, kernels.cu run_chunk_rlc), on top of the host build of the device headers
// in hostsim.cpp.  Built by tests/test_verify_all.py into a library of its own.  Test scaffolding: never linked into
// libjjschnorr_b200.so.
#include "hostsim.cpp"
#include "../../jubjub_schnorr_b200/csrc/rlc.cuh"

#include <utility>

// The combination of a list of sort entries as the kernels evaluate it: sort by key, segments of L entries and the merge levels
// of their carries, running sums over slices of `slice` buckets, Horner over the windows.
static ext rlc_msm_host(std::vector<uint32_t> keys, std::vector<uint32_t> vals, const fq* pu, const fq* pv, const RlcShape& s, int L, uint32_t slice) {
    std::vector<std::pair<uint32_t, uint32_t>> e(keys.size());
    for (size_t i = 0; i < keys.size(); i++) e[i] = {keys[i], vals[i]};
    std::sort(e.begin(), e.end(), [](const std::pair<uint32_t, uint32_t>& a, const std::pair<uint32_t, uint32_t>& b) { return a.first < b.first; });
    for (size_t i = 0; i < e.size(); i++) { keys[i] = e[i].first; vals[i] = e[i].second; }
    std::vector<ext> buckets(s.sentinel);
    for (ext& b : buckets) ext_identity(b);
    size_t len = keys.size(), segs = rlc_segments(len, L);
    std::vector<uint32_t> ck(2 * segs + 2), nk;
    std::vector<ext> cp(2 * segs + 2), np;
    for (size_t t = 0; t < segs; t++)
        rlc_segment(keys.data(), RlcAffineSrc{pu, pv, vals.data()}, len, t, L, s.sentinel, buckets.data(), ck.data(), cp.data(), segs == 1);
    while (segs > 1) {
        len = 2 * segs;
        segs = rlc_segments(len, L);
        nk.assign(2 * segs + 2, 0);
        np.assign(2 * segs + 2, ext{});
        for (size_t t = 0; t < segs; t++)
            rlc_segment(ck.data(), RlcExtSrc{cp.data()}, len, t, L, s.sentinel, buckets.data(), nk.data(), np.data(), segs == 1);
        ck.swap(nk);
        cp.swap(np);
    }
    std::vector<ext> W(s.nw_big);
    for (int w = 0; w < s.nw_big; w++) {
        ext acc;
        ext_identity(acc);
        for (uint32_t lo = 0; lo < s.buckets_per_window; lo += slice) {
            ext part;
            rlc_bucket_slice(part, &buckets[(size_t)w * s.buckets_per_window], lo, lo + slice);
            rlc_add(acc, part);
        }
        W[w] = acc;
    }
    ext P;
    rlc_horner(P, W.data(), s.nw_big, s.c);
    return P;
}

static void ext_to_wire(uint8_t* out32, const ext& P) {
    fq zi, u, v;
    fq_inv(zi, P.Z);
    fq_mul(u, P.X, zi);
    fq_mul(v, P.Y, zi);
    uint32_t w[8];
    point_to_wire(w, u, v);
    memcpy(out32, w, 32);
}

extern "C" {
void hs_chacha20_block(const uint32_t* key8, uint32_t counter, const uint32_t* nonce3, uint32_t* out16) { chacha20_block(out16, key8, counter, nonce3); }
void hs_rlc_weights(const uint8_t* seed32, uint64_t index, uint32_t* z4, uint32_t* z2_4) {
    RlcSeed seed;
    memcpy(seed.w, seed32, 32);
    rlc_weights(z4, z2_4, seed, index);
}

// sum_i k_i P_i (k_i < 2^252, 32-byte little-endian; P_i wire points that decode) through the digit, segment and bucket stages
// with window width c, L entries per segment and `slice` buckets per running-sum slice; the wire encoding of the result
int hs_rlc_msm(const uint8_t* pts32, const uint8_t* k32, size_t n, int c, int L, uint32_t slice, uint8_t* out32) {
    ensure_ready();
    if (L < 4) return -2;   // a level of segments shorter than 4 entries does not shrink its carries
    const RlcShape s = rlc_shape(0, c);
    std::vector<fq> pu(n), pv(n);
    std::vector<uint32_t> keys((size_t)s.nw_big * n), vals((size_t)s.nw_big * n);
    for (size_t i = 0; i < n; i++) {
        uint32_t w[8], k[8];
        memcpy(w, pts32 + 32 * i, 32);
        if (!point_from_wire(pu[i], pv[i], w, g_tables)) return -1;
        memcpy(k, k32 + 32 * i, 32);
        rlc_scalar_entries(&keys[(size_t)s.nw_big * i], &vals[(size_t)s.nw_big * i], k, s.nw_big, s, (uint32_t)i, false);
    }
    ext P = rlc_msm_host(keys, vals, pu.data(), pv.data(), s, L, slice);
    ext_to_wire(out32, P);
    return 0;
}

// jjs_verify_all through the stages of run_chunk_rlc, in one pass: decode with every point subgroup-tested, hash of the items
// whose keys are valid, validity by the reference's precedence, entries and G scalars, the combination, the G terms, the check
void hs_verify_all(int variant, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg, size_t n, const uint8_t* seed32, int c, int L, int* all_valid) {
    ensure_ready();
    const int slots = variant_slots(variant);
    const bool dbl = variant == VAR_DOUBLE;
    const uint32_t pks = dbl ? 64 : 32, sgs = dbl ? 96 : 64;
    RlcSeed seed;
    memcpy(seed.w, seed32, 32);
    const RlcShape s = rlc_shape(dbl, c);
    std::vector<fq> pu(slots * n), pv(slots * n);
    std::vector<uint8_t> pf(slots * n), itf(n);
    std::vector<uint32_t> cw(8 * n), keys((size_t)s.per_item * n), vals((size_t)s.per_item * n), zu(16 * n);
    WireField fmsg{msg, 32}, fu{sig, sgs};
    for (int sl = 0; sl < slots; sl++) {
        const WireField f = dbl ? (sl < 2 ? WireField{pk + 32 * sl, pks} : WireField{sig + 32 * (sl - 1), sgs})
                                : (sl == 0 ? WireField{pk, pks} : WireField{sig + 32, sgs});
        for (size_t i = 0; i < n; i++) stage_decode(f, i, pu.data(), pv.data(), pf.data(), sl * n + i, g_tables, true);
    }
    bool valid = true;
    uint32_t su[2][8] = {{0}};
    for (size_t i = 0; i < n; i++) {
        stage_challenge(variant, pu.data(), pv.data(), pf.data(), n, i, fmsg, fu, cw.data(), itf.data());
        const bool ok = stage_status(variant, pf.data(), (uint8_t)(itf[i] | IF_EQ0_OK | IF_EQ1_OK), n, i) == 0;
        valid = valid && ok;
        uint32_t u[8];
        wire_load(u, fu, i);
        rlc_item_entries(&keys[(size_t)s.per_item * i], &vals[(size_t)s.per_item * i], &zu[8 * i], &zu[8 * (n + i)], dbl, ok, &cw[8 * i], u, seed, i, n,
                         i, s);
        fr_add(su[0], su[0], &zu[8 * i]);
        if (dbl) fr_add(su[1], su[1], &zu[8 * (n + i)]);
    }
    ext P = n ? rlc_msm_host(keys, vals, pu.data(), pv.data(), s, L, 32) : ext{};
    if (!n) ext_identity(P);
    rlc_fixed_terms<FB_W>(P, su, dbl, g_tables.fb_g, g_tables.fb_gn);
    *all_valid = valid && ext_is_identity(P) ? 1 : 0;
}
}
