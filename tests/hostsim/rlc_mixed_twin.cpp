// CPU twin of whole-batch verification over the parts of a mixed call (jjs_verify_all_mixed: csrc/rlc.cuh, kernels.cu
// run_chunk_rlc), on top of rlc_twin.cpp and the host simulator.  Built by tests/test_verify_all_mixed.py into a library of its
// own.  Test scaffolding: never linked into libjjschnorr_b200.so.
#include "rlc_twin.cpp"

extern "C" {
// jjs_verify_all_mixed through the stages of run_chunk_rlc, every part in one pass: decode with every point subgroup-tested
// (aggregate parts: signer keys decoded, aggregation by stage_aggregate_coeffs / stage_aggregate as hs_verify_aggregate runs it,
// R decoded with its test), the hash of the items whose keys are valid, validity by the reference's precedence, entries and G
// scalars with the weights of the item's position in the whole call, one combination over every part's entries, the G and G'
// terms, the check.  Part p: kind kinds[p] (JJS_KIND_*), ns[p] items, wire buffers pks[p] / sigs[p] / msgs[p], offsets[p]
// (n + 1 entries, aggregate parts only).
void hs_verify_all_mixed(size_t n_parts, const int* kinds, const uint8_t* const* pks, const uint8_t* const* sigs, const uint8_t* const* msgs,
                         const uint32_t* const* offsets, const size_t* ns, const uint8_t* seed32, int c, int L, int* all_valid) {
    ensure_ready();
    RlcSeed seed;
    memcpy(seed.w, seed32, 32);
    const RlcShape s0 = rlc_shape(VAR_SINGLE, c);   // sentinel and windows do not depend on the kind
    std::vector<fq> pu, pv;                          // the points of every part, part after part
    std::vector<uint32_t> keys, vals;
    bool valid = true;
    uint32_t su[2][8] = {{0}};
    uint64_t base = 0;
    for (size_t p = 0; p < n_parts; p++) {
        const size_t n = ns[p];
        const bool agg = kinds[p] == 3;   // JJS_KIND_AGGREGATE; the other kinds are the variants
        const int variant = agg ? VAR_SINGLE : kinds[p], slots = variant_slots(variant);
        const bool dbl = variant == VAR_DOUBLE;
        const uint32_t pks_ = variant == VAR_SINGLE ? 32 : 64, sgs = dbl ? 96 : 64;
        const RlcShape s = rlc_shape(variant, c);
        std::vector<fq> qu(slots * n), qv(slots * n);
        std::vector<uint8_t> pf(slots * n), itf(n);
        std::vector<uint32_t> cw(8 * n), zu(16 * n);
        WireField fmsg{msgs[p], 32}, fu{sigs[p], sgs};
        if (agg) {
            const uint32_t* off = offsets[p];
            const size_t K = off[n] - off[0];
            std::vector<fq> ku(K + 1), kv(K + 1), tab(R32_TAB_FQ * AGG_GROUP);
            std::vector<uint8_t> kf(K + 1);
            std::vector<uint32_t> kc(8 * K + 8);
            size_t max_cnt = 0;
            for (size_t i = 0; i < n; i++) max_cnt = std::max<size_t>(max_cnt, off[i + 1] - off[i]);
            const fq* tags = tags_upto(2 + 2 * max_cnt);
            for (size_t k = 0; k < K; k++) stage_decode(WireField{pks[p], 32}, off[0] + k, ku.data(), kv.data(), kf.data(), k, g_tables, false);
            for (size_t i = 0; i < n; i++) {
                const uint32_t lo = off[i] - off[0], hi = off[i + 1] - off[0];
                stage_aggregate_coeffs(ku.data(), kv.data(), kf.data(), lo, hi, kc.data(), tags);
                uint32_t w[8];
                stage_aggregate(ku.data(), kv.data(), kf.data(), lo, hi, qu.data(), qv.data(), pf.data(), i, w, tab.data(), 1, tags, kc.data());
                stage_decode(WireField{sigs[p] + 32, 64}, i, qu.data(), qv.data(), pf.data(), n + i, g_tables, true);
            }
        } else {
            for (int sl = 0; sl < slots; sl++) {
                WireField f;
                if (variant == VAR_SINGLE) f = sl == 0 ? WireField{pks[p], pks_} : WireField{sigs[p] + 32, sgs};
                else if (variant == VAR_DOUBLE) f = sl < 2 ? WireField{pks[p] + 32 * sl, pks_} : WireField{sigs[p] + 32 * (sl - 1), sgs};
                else f = sl < 2 ? WireField{pks[p] + 32 * sl, pks_} : WireField{sigs[p] + 32, sgs};
                for (size_t i = 0; i < n; i++) stage_decode(f, i, qu.data(), qv.data(), pf.data(), sl * n + i, g_tables, true);
            }
        }
        const size_t k0 = keys.size(), point_base = pu.size();
        keys.resize(k0 + (size_t)s.per_item * n);
        vals.resize(k0 + (size_t)s.per_item * n);
        for (size_t i = 0; i < n; i++) {
            stage_challenge(variant, qu.data(), qv.data(), pf.data(), n, i, fmsg, fu, cw.data(), itf.data());
            const bool ok = stage_status(variant, pf.data(), (uint8_t)(itf[i] | IF_EQ0_OK | IF_EQ1_OK), n, i) == 0;
            valid = valid && ok;
            uint32_t u[8];
            wire_load(u, fu, i);
            uint32_t* k = &keys[k0 + (size_t)s.per_item * i];
            uint32_t* v = &vals[k0 + (size_t)s.per_item * i];
            rlc_item_entries(k, v, &zu[8 * i], &zu[8 * (n + i)], variant, ok, &cw[8 * i], u, seed, base + i, n, i, s);
            for (int e = 0; e < s.per_item; e++) v[e] += 2 * (uint32_t)point_base;   // references into the joint point arrays
            fr_add(su[0], su[0], &zu[8 * i]);
            if (dbl) fr_add(su[1], su[1], &zu[8 * (n + i)]);
        }
        pu.insert(pu.end(), qu.begin(), qu.end());
        pv.insert(pv.end(), qv.begin(), qv.end());
        base += n;
    }
    ext P;
    if (keys.empty()) ext_identity(P);
    else P = rlc_msm_host(keys, vals, pu.data(), pv.data(), s0, L, 32);
    rlc_fixed_terms<FB_W>(P, su, true, g_tables.fb_g, g_tables.fb_gn);
    *all_valid = valid && ext_is_identity(P) ? 1 : 0;
}
}
