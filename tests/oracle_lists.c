/* oracle_lists.c -- TEST INFRASTRUCTURE ONLY: BaseType(row, min_af) + lrt(list) of one site over an ordered candidate list,
 * restated on the CPU for the tests of the list kernel (K8).  It is compiled together with the oracle (oracle/bv_oracle.c is
 * included, so the list path runs the very lrt_core, Fisher and chi-square code that bvo_site / bvo_group_site run) into a
 * library of its own; tests/oracle_lists.py builds and loads it.  Nothing under basevar_b200/ uses it. */
#include "../oracle/bv_oracle.c"

/* ------------------------------------------------------------------------------------------------
 * BaseType(bi, min_af) + lrt(list) of one site over an ORDERED candidate list (src/basetype.h:117-118,
 * src/basetype.cpp:130-199): lrt_core over `list`, then ALT in list order, QUAL (:180-194) with the first active
 * base in list order, and FS of strand_bias(REF, ALT set) (:244-295).  Entries after the n_list-th are ignored.
 * Returns -1 (output all-zero) for a repeated base or a code outside 0..3.
 * ------------------------------------------------------------------------------------------------ */
int bvo_site_list(const uint8_t* base, const uint8_t* qual, const uint8_t* strand, uint32_t n_samples, uint8_t ref_char,
                  const uint8_t* list, int n_list, const bv_params* prm, bv_lrt_out* out) {
    memset(out, 0, sizeof(*out));
    int cand[4], seen = 0;
    if (n_list < 0 || n_list > 4) return -1;
    for (int k = 0; k < n_list; ++k) {
        if (list[k] > 3 || (seen >> list[k] & 1)) return -1;
        seen |= 1 << list[k];
        cand[k] = list[k];
    }
    if (n_list == 0) return 0;
    double* lik = (double*)malloc(sizeof(double) * 4 * (size_t)(n_samples ? n_samples : 1));
    size_t d = 0;
    double depth[4] = {0, 0, 0, 0};
    int fwd[4] = {0, 0, 0, 0}, rev[4] = {0, 0, 0, 0};
    unsigned flags = 0;
    for (uint32_t i = 0; i < n_samples; ++i) { /* BaseType::BaseType, src/basetype.cpp:45-71 */
        uint8_t b = base[i];
        if (b >= BV_BASE_N) continue;
        uint8_t q = qual[i];
        if (q > BV_QUAL_MAX) flags |= BV_FLAG_BAD_QUAL;
        double eps = exp((double)q * kMLN10TO10);
        if (b < 4) {
            depth[b] += 1;
            if (strand[i] == BV_STRAND_FWD) fwd[b]++;
            else if (strand[i] == BV_STRAND_REV) rev[b]++;
        }
        if (strand[i] != BV_STRAND_FWD && strand[i] != BV_STRAND_REV) flags |= BV_FLAG_BAD_STRAND;
        for (int j = 0; j < 4; ++j) lik[4 * d + j] = (b == j) ? 1.0 - eps : eps / 3;
        ++d;
    }
    const int total = (int)d;
    if (total == 0) { free(lik); return 0; }
    int up_ref = ref_char;
    if (up_ref >= 'a' && up_ref <= 'z') up_ref -= 32;
    int ref_code = up_ref == 'A' ? 0 : up_ref == 'C' ? 1 : up_ref == 'G' ? 2 : up_ref == 'T' ? 3 : -1;
    lrt_result res;
    int n_active = lrt_core(lik, d, depth, total, cand, n_list, prm, &flags, &res);
    free(lik);
    if (n_active == 0) {
        out->flags = (uint8_t)flags;
        return 0;
    }
    int rf = 0, rr = 0, af_ = 0, ar = 0;
    if (ref_code >= 0) { rf = fwd[ref_code]; rr = rev[ref_code]; }
    for (int k = 0; k < n_active; ++k) {
        if (res.active[k] != ref_code) {
            out->alt[out->n_alt] = (uint8_t)res.active[k];
            out->af[out->n_alt] = res.f_act[res.active[k]];
            af_ += fwd[res.active[k]]; ar += rev[res.active[k]];
            out->n_alt++;
        }
    }
    out->n_active = (uint8_t)n_active;
    out->chi2 = res.chi;
    out->em_calls = (uint8_t)res.em_calls;
    if (out->n_alt) {
        double r = depth[res.active[0]] / (double)total;
        if (n_active == 1 && total > 10 && r > 0.5) {
            out->qual = 5000.0;
            flags |= BV_FLAG_MONO_QUAL;
        } else {
            double p = bvo_chi2_test(res.chi, 1);
            if (isnan(p)) p = 1.0;
            double qv = (p != 0.0) ? -10 * log10(p) : 10000.0;
            if (qv == -0.0) qv = 0.0;
            out->qual = qv;
        }
        out->fs = bvo_fs_from_table(rf, rr, af_, ar);
    }
    out->flags = (uint8_t)flags;
    return 0;
}
