// CPU twin of grouped verification (jjs_verify_grouped: csrc/rlc.cuh, kernels.cu run_chunk_rlc with a GroupedOut), on top of
// rlc_mixed_twin.cpp and the host simulator.  Built by tests/test_verify_grouped.py into a library of its own.  Test
// scaffolding: never linked into libjjschnorr_b200.so.
#include "rlc_mixed_twin.cpp"

// The combination of every group of a pass as the kernels evaluate it: the sort entries carry grouped keys, so one sort, one
// segment pass and one bucket array serve all groups; the running sums run over groups x nw_big windows and Horner over each
// group's windows.
static std::vector<ext> rlc_msm_groups_host(std::vector<uint32_t> keys, std::vector<uint32_t> vals, const fq* pu, const fq* pv, const RlcShape& s,
                                            size_t groups, int L, uint32_t slice) {
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
    const size_t nwin = groups * (size_t)s.nw_big;
    std::vector<ext> W(nwin), out(groups);
    for (size_t w = 0; w < nwin; w++) {
        ext acc;
        ext_identity(acc);
        for (uint32_t lo = 0; lo < s.buckets_per_window; lo += slice) {
            ext part;
            rlc_bucket_slice(part, &buckets[w * s.buckets_per_window], lo, lo + slice);
            rlc_add(acc, part);
        }
        W[w] = acc;
    }
    for (size_t grp = 0; grp < groups; grp++) rlc_horner(out[grp], &W[grp * s.nw_big], s.nw_big, s.c);
    return out;
}

static bool ext_equal(const ext& a, const ext& b) {
    fq l, r;
    fq_mul(l, a.X, b.Z);
    fq_mul(r, b.X, a.Z);
    if (memcmp(l.l, r.l, 32) != 0) return false;
    fq_mul(l, a.Y, b.Z);
    fq_mul(r, b.Y, a.Z);
    return memcmp(l.l, r.l, 32) == 0;
}

extern "C" {
// jjs_verify_grouped through the stages of the grouped pass, every part in one pass of groups of g consecutive items: the front
// of hs_verify_all_mixed (every point subgroup-tested), validity by the reference's precedence, grouped entries and per-group G
// scalars with the weights of the item's position in the whole call, one combination per group, the verdicts, then the
// per-item equations (hostsim's equation_with_rtest) for the valid items of failing groups, statuses and challenges as
// k_finalize writes them.  Arguments as hs_verify_all_mixed; outputs, all parts concatenated: status[item], c32[item],
// verdict[group] (groups of every part, part after part), *fallback = items verified one by one.  Returns the number of groups,
// or -1 if a one-group pass's point differs from the whole-batch combination of the same entries.
long hs_verify_grouped(size_t n_parts, const int* kinds, const uint8_t* const* pks, const uint8_t* const* sigs, const uint8_t* const* msgs,
                       const uint32_t* const* offsets, const size_t* ns, const uint8_t* seed32, size_t g, int c, int L, uint8_t* status, uint8_t* c32,
                       uint8_t* verdict, uint64_t* fallback) {
    ensure_ready();
    RlcSeed seed;
    memcpy(seed.w, seed32, 32);
    uint64_t base = 0;
    size_t groups_done = 0;
    *fallback = 0;
    for (size_t p = 0; p < n_parts; p++) {
        const size_t n = ns[p];
        if (!n) continue;
        const bool agg = kinds[p] == 3;   // JJS_KIND_AGGREGATE; the other kinds are the variants
        const int variant = agg ? VAR_SINGLE : kinds[p], slots = variant_slots(variant);
        const bool dbl = variant == VAR_DOUBLE;
        const uint32_t pks_ = variant == VAR_SINGLE ? 32 : 64, sgs = dbl ? 96 : 64;
        const size_t G = (n + g - 1) / g;
        const RlcShape s = rlc_shape(variant, c, G);
        std::vector<fq> qu(slots * n), qv(slots * n), tab(108);
        std::vector<uint8_t> pf(slots * n), itf(n), ok(n);
        std::vector<uint32_t> cw(8 * n), zu(16 * n), keys((size_t)s.per_item * n), vals((size_t)s.per_item * n);
        WireField fmsg{msgs[p], 32}, fu{sigs[p], sgs};
        if (agg) {
            const uint32_t* off = offsets[p];
            const size_t K = off[n] - off[0];
            std::vector<fq> ku(K + 1), kv(K + 1), atab(R32_TAB_FQ * AGG_GROUP);
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
                stage_aggregate(ku.data(), kv.data(), kf.data(), lo, hi, qu.data(), qv.data(), pf.data(), i, w, atab.data(), 1, tags, kc.data());
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
        std::vector<uint32_t> su(16 * G, 0);
        for (size_t i = 0; i < n; i++) {
            stage_challenge(variant, qu.data(), qv.data(), pf.data(), n, i, fmsg, fu, cw.data(), itf.data());
            ok[i] = stage_status(variant, pf.data(), (uint8_t)(itf[i] | IF_EQ0_OK | IF_EQ1_OK), n, i) == 0;
            uint32_t u[8];
            wire_load(u, fu, i);
            rlc_item_entries(&keys[(size_t)s.per_item * i], &vals[(size_t)s.per_item * i], &zu[8 * i], &zu[8 * (n + i)], variant, ok[i], &cw[8 * i], u, seed,
                             base + i, n, i, s, (uint32_t)(i / g));
            uint32_t* sg = &su[16 * (i / g)];
            fr_add(sg, sg, &zu[8 * i]);
            if (dbl) fr_add(sg + 8, sg + 8, &zu[8 * (n + i)]);
        }
        const std::vector<ext> P = rlc_msm_groups_host(keys, vals, qu.data(), qv.data(), s, G, L, 32);
        if (G == 1 && !ext_equal(P[0], rlc_msm_host(keys, vals, qu.data(), qv.data(), rlc_shape(variant, c), L, 32))) return -1;
        for (size_t grp = 0; grp < G; grp++) {
            ext Q = P[grp];
            rlc_fixed_terms<FB_W>(Q, reinterpret_cast<const uint32_t(*)[8]>(&su[16 * grp]), true, g_tables.fb_g, g_tables.fb_gn);
            verdict[groups_done + grp] = ext_is_identity(Q) ? 1 : 0;
        }
        for (size_t i = 0; i < n; i++) {
            uint8_t fl = itf[i];
            if (ok[i] && verdict[groups_done + i / g]) {
                fl |= IF_EQ0_OK | IF_EQ1_OK;
            } else if (ok[i]) {
                (*fallback)++;
                for (int eq = 0; eq < (dbl ? 2 : 1); eq++)
                    if (equation_with_rtest(variant, eq, qu.data(), qv.data(), pf.data(), n, i, fu, cw.data(), tab.data())) fl |= eq ? IF_EQ1_OK : IF_EQ0_OK;
            }
            const uint8_t st = stage_status(variant, pf.data(), fl, n, i);
            status[base + i] = st;
            if (st <= 1) memcpy(c32 + 32 * (base + i), &cw[8 * i], 32);
            else memset(c32 + 32 * (base + i), 0, 32);
        }
        groups_done += G;
        base += n;
    }
    return (long)groups_done;
}
}
