// CPU twin of key sets at every key-window width (csrc/keyset.cuh: KW = 8..4 and points only, the layouts of
// jjs_keyset_create_limited), on top of the host build of the device headers in hostsim.cpp (its tables, its equation counters
// and all of its hs_* entry points are part of this library too).  The width is taken at run time and dispatched through
// with_key_width, as the library does.  Built by tests/test_keyset_limited.py into a library of its own.  Test scaffolding:
// never linked into libjjschnorr_b200.so.
#include "hostsim.cpp"
#include "../../jubjub_schnorr_b200/csrc/keyset.cuh"

// The twin's registered key set (one at a time): decoded key points slot-major, their flags, and the window tables of width
// key_bits key-major (none for key_bits 0, a points-only set), laid out as the library lays them out on a device.
static struct {
    int variant = VAR_SINGLE;
    int key_bits = KEYED_W;
    size_t n_keys = 0;
    std::vector<fq> u, v;
    std::vector<uint8_t> flags;
    std::vector<niels> table;
} g_ks;

extern "C" {
// jjs_keyset_create (key_bits 8) and jjs_keyset_create_limited on the twin: decode with the subgroup test, then, unless
// key_bits is 0, the two table passes of k_keyset_bases / k_keyset_combine at that width
void hs_keyset_build_w(int variant, int key_bits, const uint8_t* pk, size_t n_keys, uint8_t* key_status) {
    ensure_ready();
    const int nk = keyed_points(variant);
    const size_t npts = (size_t)nk * n_keys;
    g_ks.variant = variant;
    g_ks.key_bits = key_bits;
    g_ks.n_keys = n_keys;
    g_ks.u.assign(npts, fq{});
    g_ks.v.assign(npts, fq{});
    g_ks.flags.assign(npts, 0);
    g_ks.table.clear();
    for (int s = 0; s < nk; s++)
        for (size_t k = 0; k < n_keys; k++)
            stage_decode(WireField{pk + 32 * s, (uint32_t)(32 * nk)}, k, g_ks.u.data(), g_ks.v.data(), g_ks.flags.data(), s * n_keys + k, g_tables, true);
    if (key_bits)
        with_key_width(key_bits, [&](auto kwc) {
            constexpr int KW = decltype(kwc)::value, WINDOWS = keyed_windows(KW), ENTRIES = keyed_entries(KW), PE = keyed_point_entries(KW);
            g_ks.table.assign(npts * PE, niels{});
            std::vector<ext> bases(WINDOWS);
            for (size_t p = 0; p < npts; p++) {
                const size_t k = (p % nk) * n_keys + p / nk;
                fq bu, bv;
                keyed_table_base(bu, bv, g_ks.u[k], g_ks.v[k], g_ks.flags[k]);
                keyed_window_bases<KW>(bases.data(), 1, bu, bv);
                for (int w = 0; w < WINDOWS; w++)
                    for (int g = 0; g < ENTRIES / KEYED_BATCH; g++)
                        keyed_combine_entries<KW>(&g_ks.table[p * PE + (size_t)w * ENTRIES + (size_t)g * KEYED_BATCH], bases[w], g * KEYED_BATCH + 1);
            }
        });
    for (size_t k = 0; k < n_keys; k++) key_status[k] = keyed_key_status(variant, g_ks.flags.data(), n_keys, k);
}
// entry (w, j) of key point p (key * points_per_key + point) from its definition (keyed_table_entry) and as built, at the set's width
void hs_keyed_entry(size_t p, int w, int j, uint32_t* out24, uint32_t* ref24) {
    const int nk = keyed_points(g_ks.variant);
    const size_t k = (p % nk) * g_ks.n_keys + p / nk;
    fq bu, bv;
    keyed_table_base(bu, bv, g_ks.u[k], g_ks.v[k], g_ks.flags[k]);
    niels e;
    with_key_width(g_ks.key_bits, [&](auto kwc) {
        constexpr int KW = decltype(kwc)::value;
        keyed_table_entry<KW>(e, bu, bv, w, j);
        memcpy(ref24, &g_ks.table[p * keyed_point_entries(KW) + (size_t)w * keyed_entries(KW) + (size_t)(j - 1)], 96);
    });
    memcpy(out24, &e, 96);
}
// jjs_verify_keyed through the stage functions of run_chunk_keyed: gather, signature points decoded with the test deferred,
// hash, keyed equations (per-item equations under a points-only set, as run_chunk) and the deferred tests they ask for, status
void hs_verify_keyed(const uint32_t* key_index, const uint8_t* sig, const uint8_t* msg, size_t n, uint8_t* status, uint8_t* c_out) {
    ensure_ready();
    const int variant = g_ks.variant, nk = keyed_points(variant), slots = variant_slots(variant);
    const uint32_t sgs = variant == VAR_DOUBLE ? 96 : 64;
    std::vector<fq> pu(slots * n), pv(slots * n), tab(108);
    std::vector<uint8_t> pf(slots * n), itf(n);
    std::vector<uint32_t> cw(8 * n);
    WireField fmsg{msg, 32}, fu{sig, sgs};
    for (size_t i = 0; i < n; i++)
        stage_keyed_gather(variant, g_ks.u.data(), g_ks.v.data(), g_ks.flags.data(), g_ks.n_keys, key_index[i], pu.data(), pv.data(), pf.data(), n, i);
    for (int s = 0; s < nk; s++)
        for (size_t i = 0; i < n; i++) stage_decode(WireField{sig + 32 + 32 * s, sgs}, i, pu.data(), pv.data(), pf.data(), (nk + s) * n + i, g_tables, false);
    for (size_t i = 0; i < n; i++) {
        if (stage_challenge(variant, pu.data(), pv.data(), pf.data(), n, i, fmsg, fu, cw.data(), itf.data())) {
            for (int eq = 0; eq < nk; eq++) {
                bool ok;
                if (g_ks.key_bits == 0) {
                    ok = equation_with_rtest(variant, eq, pu.data(), pv.data(), pf.data(), n, i, fu, cw.data(), tab.data());
                } else {
                    bool need = false;
                    ok = with_key_width(g_ks.key_bits, [&](auto kwc) {
                        constexpr int KW = decltype(kwc)::value;
                        const niels* ktab = &g_ks.table[((size_t)key_index[i] * nk + eq) * keyed_point_entries(KW)];
                        return stage_equation_keyed<FB_W, KW>(variant, eq, pu.data(), pv.data(), pf.data(), n, i, eq ? g_tables.fb_gn : g_tables.fb_g, ktab,
                                                              fu, cw.data(), &need);
                    });
                    g_equations++;
                    if (need) {
                        int pk_slot, r_slot, base_slot;
                        equation_slots(variant, eq, pk_slot, r_slot, base_slot);
                        stage_rtest(pu.data(), pv.data(), pf.data(), (size_t)r_slot * n + i);
                        g_rtests++;
                    }
                }
                if (ok) itf[i] |= eq ? IF_EQ1_OK : IF_EQ0_OK;
            }
        }
        status[i] = stage_status(variant, pf.data(), itf[i], n, i);
        if (status[i] <= 1) memcpy(c_out + 32 * i, &cw[8 * i], 32); else memset(c_out + 32 * i, 0, 32);
    }
}
}
