// TEST-ONLY host build of the registered-key-set path (schnorr-sig_b200/csrc/keyset.cuh) with g++, for
// tests/test_registered_hostsim.py.  It extends the host build of the device headers (hostsim.cpp, included whole:
// the same G table, counters and helpers) with the exports below; like it, it is not part of the product.
#include "hostsim.cpp"
#include "../../schnorr-sig_b200/csrc/keyset.cuh"

// ---- registered key sets (keyset.cuh) ----
API void hs_kt_geometry(int* w, int* windows, int* entries) {
    *w = KT_W;
    *windows = KT_WINDOWS;
    *entries = KT_ENTRIES;
}
// signed-window table of the affine point p96 through the builder the kernels run (tab_bases + tab_entry):
// out = windows x (2^(w-1) + 1) x 12 limbs
API void hs_tab_build(const uint8_t* p96, int w, int windows, uint64_t* out) {
    uint64_t pt[12];
    memcpy(pt, p96, 96);
    std::vector<jac_pt> bases(windows);
    tab_bases(pt, w, windows, bases.data());
    int entries = (1 << (w - 1)) + 1;
    for (int i = 0; i < windows; i++)
        for (int d = 0; d < entries; d++) tab_entry(bases[i], w, d, out + ((size_t)i * entries + d) * 12);
}
API int hs_keyset_key_status(const uint8_t* p96, int inf) {
    uint64_t pt[12];
    memcpy(pt, p96, 96);
    jac_pt d;
    return keyset_key_status(pt, inf != 0, &d);
}
// h*P + e*G from a key table (hs_tab_build at KT_W) and the G table: fast_result; out96 = the affine result unless
// FAST_EXCEPTIONAL
API int hs_verify_core_reg(const uint64_t* ktab, const uint8_t* h32, const uint8_t* e32, uint8_t* out96) {
    build_gtab();
    jf_pt r;
    int fr = verify_core_reg(ldsc(h32), ldsc(e32), ktab, g_gtab.data(), &r);
    if (fr != FAST_EXCEPTIONAL) jf_to_affine(r, out96);
    return fr;
}
// full per-signature path as k_keyset_register + k_keyset_gather + k_ingest + k_verify_reg (+ k_verify for the items
// handed back) compose it for a key with registration status `status` (hs_keyset_key_status) and table `ktab` (unused
// unless the status is 0 and the key is not the identity); *used_exact reports whether the exact routine ran
API int hs_verify_one_reg(const uint8_t* sig81, const uint8_t* pk96, int pk_inf, int status, const uint64_t* ktab,
                          const uint8_t* msg, uint64_t len, int* used_exact) {
    build_gtab();
    *used_exact = 0;
    fp6 sx, px, py;
    memcpy(sx.c, sig81, 48);
    memcpy(px.c, pk96, 48);
    memcpy(py.c, pk96 + 48, 48);
    scalar e = ldsc(sig81 + 49);
    bool x_ok = fp6_is_canonical(sx);
    if (status == KEY_MALFORMED || sc_geq_q(e)) return VERDICT_MALFORMED;   // k_ingest's malformed flag
    scalar h = sc_zero();
    if (!pk_inf) {
        uint8_t v = VERDICT_INVALID_PUBLIC_KEY;
        if (status == KEY_OK) {
            if (x_ok) h = challenge_scalar(sx, px, py, false, msg, len);
            jf_pt r;
            int fr = verify_core_reg(h, e, ktab, g_gtab.data(), &r);
            v = reg_verdict((uint8_t)status, x_ok, fr, r, sx);
        }
        if (v != VERDICT_NEEDS_EXACT) return v;
    }
    *used_exact = 1;
    if (x_ok) h = challenge_scalar(sx, px, py, pk_inf != 0, msg, len);
    jac_pt d;
    return verify_points(sx, x_ok, e, px, py, pk_inf != 0, h, g_gtab.data(), &d);
}

