// CPU twin of verification against registered key sets (csrc/keyset.cuh), on top of the host build of the device headers in
// hostsim.cpp (its tables, its equation counters and all of its hs_* entry points are part of this library too).  Built by
// tests/test_keyset.py into a library of its own.  Test scaffolding: never linked into libjjschnorr_b200.so.
#include "hostsim.cpp"
#include "../../jubjub_schnorr_b200/csrc/keyset.cuh"

// The twin's registered key set (one at a time): decoded key points slot-major, their flags, and the window tables key-major,
// laid out as the library lays them out on a device.
static struct {
    int variant = VAR_SINGLE;
    size_t n_keys = 0;
    std::vector<fq> u, v;
    std::vector<uint8_t> flags;
    std::vector<niels> table;
} g_ks;

extern "C" {
// jjs_keyset_create on the twin: decode with the subgroup test, then the two table passes of k_keyset_bases / k_keyset_combine
void hs_keyset_build(int variant, const uint8_t* pk, size_t n_keys, uint8_t* key_status) {
    ensure_ready();
    const int nk = keyed_points(variant);
    const size_t npts = (size_t)nk * n_keys;
    g_ks.variant = variant;
    g_ks.n_keys = n_keys;
    g_ks.u.assign(npts, fq{});
    g_ks.v.assign(npts, fq{});
    g_ks.flags.assign(npts, 0);
    g_ks.table.assign(npts * KEYED_POINT_ENTRIES, niels{});
    for (int s = 0; s < nk; s++)
        for (size_t k = 0; k < n_keys; k++)
            stage_decode(WireField{pk + 32 * s, (uint32_t)(32 * nk)}, k, g_ks.u.data(), g_ks.v.data(), g_ks.flags.data(), s * n_keys + k, g_tables, true);
    std::vector<ext> bases(KEYED_WINDOWS);
    for (size_t p = 0; p < npts; p++) {
        const size_t k = (p % nk) * n_keys + p / nk;
        fq bu, bv;
        keyed_table_base(bu, bv, g_ks.u[k], g_ks.v[k], g_ks.flags[k]);
        keyed_window_bases(bases.data(), 1, bu, bv);
        for (int w = 0; w < KEYED_WINDOWS; w++)
            for (int g = 0; g < KEYED_ENTRIES / KEYED_BATCH; g++)
                keyed_combine_entries(&g_ks.table[p * KEYED_POINT_ENTRIES + (size_t)w * KEYED_ENTRIES + (size_t)g * KEYED_BATCH], bases[w], g * KEYED_BATCH + 1);
    }
    for (size_t k = 0; k < n_keys; k++) key_status[k] = keyed_key_status(variant, g_ks.flags.data(), n_keys, k);
}
// entry (w, j) of key point p (key * points_per_key + point) from its definition (keyed_table_entry) and as built
void hs_keyed_entry(size_t p, int w, int j, uint32_t* out24, uint32_t* ref24) {
    const int nk = keyed_points(g_ks.variant);
    const size_t k = (p % nk) * g_ks.n_keys + p / nk;
    fq bu, bv;
    keyed_table_base(bu, bv, g_ks.u[k], g_ks.v[k], g_ks.flags[k]);
    niels e;
    keyed_table_entry(e, bu, bv, w, j);
    memcpy(out24, &e, 96);
    memcpy(ref24, &g_ks.table[p * KEYED_POINT_ENTRIES + (size_t)w * KEYED_ENTRIES + (size_t)(j - 1)], 96);
}
// jjs_verify_keyed through the stage functions of run_chunk_keyed: gather, signature points decoded with the test deferred,
// hash, keyed equations and the deferred tests they ask for, status
void hs_verify_keyed(const uint32_t* key_index, const uint8_t* sig, const uint8_t* msg, size_t n, uint8_t* status, uint8_t* c_out) {
    ensure_ready();
    const int variant = g_ks.variant, nk = keyed_points(variant), slots = variant_slots(variant);
    const uint32_t sgs = variant == VAR_DOUBLE ? 96 : 64;
    std::vector<fq> pu(slots * n), pv(slots * n);
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
                bool need;
                const niels* ktab = &g_ks.table[((size_t)key_index[i] * nk + eq) * KEYED_POINT_ENTRIES];
                bool ok = stage_equation_keyed(variant, eq, pu.data(), pv.data(), pf.data(), n, i, eq ? g_tables.fb_gn : g_tables.fb_g, ktab, fu, cw.data(), &need);
                g_equations++;
                if (need) {
                    int pk_slot, r_slot, base_slot;
                    equation_slots(variant, eq, pk_slot, r_slot, base_slot);
                    stage_rtest(pu.data(), pv.data(), pf.data(), (size_t)r_slot * n + i);
                    g_rtests++;
                }
                if (ok) itf[i] |= eq ? IF_EQ1_OK : IF_EQ0_OK;
            }
        }
        status[i] = stage_status(variant, pf.data(), itf[i], n, i);
        if (status[i] <= 1) memcpy(c_out + 32 * i, &cw[8 * i], 32); else memset(c_out + 32 * i, 0, 32);
    }
}
}
