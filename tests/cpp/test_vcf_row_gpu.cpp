// GPU test of the VCF row's batch path in the C++ host mirror (INTEGRATION.md section 2): sites packed with SparsePacker
// (compact results, called-site kernels, population groups through Context::set_groups) and with TilePacker (its rpr plane
// feeding ReadPosRankSum), collected with Context::wait_calls; [REF, ALT...] lists of the called sites through
// Context::submit_lists on the sparse tile with compact results.  For every site of the SURVEY.md 8c vectors and of a synthetic
// tile the batch results must equal the per-site drop-in route: BaseType(&bi, min_af).lrt() and strand_bias for the getters,
// (int) ref_vs_alt_ranksumtest(...) for the three rank sums, BaseType(&group_bi, min_af).lrt([REF, ALT...]) for every group;
// the group AFs also match the oracle's bvo_group_site.
// TEST INFRASTRUCTURE: loads the oracle library (oracle/libbvoracle.so; its path is the first argument) through dlopen; the
// host library itself never touches it.
#include <dlfcn.h>

#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../basevar_b200/host/bv_host.hpp"

using namespace bvhost;

static int g_fail = 0;
#define CHECK(cond)                                                        \
    do {                                                                   \
        if (!(cond)) { printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); ++g_fail; } \
    } while (0)

typedef int (*group_fn)(const uint8_t*, const uint8_t*, uint32_t, const uint8_t*, uint32_t, uint8_t, const uint8_t*, int,
                        const bv_params*, bv_group_out*);
static group_fn bvo_group_site = nullptr;

static bool close_rel(double a, double b, double rtol) {
    if (std::isnan(a) && std::isnan(b)) return true;
    return a == b || std::fabs(a - b) <= 1e-300 + rtol * std::fabs(b);
}
static bool same_f64(double a, double b) { return (std::isnan(a) && std::isnan(b)) || memcmp(&a, &b, 8) == 0; }
static int code_of(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }

static uint32_t g_x = 2463534242u;
static uint32_t rnd() { g_x ^= g_x << 13; g_x ^= g_x >> 17; g_x ^= g_x << 5; return g_x; }

// a site of n samples: coverage cov, REF ref, ALT reads of the bases in `alts` at fraction alt_frac each
static BatchInfo make_site(uint32_t n, char ref, const std::string& alts, double cov, double alt_frac, uint32_t pos) {
    BatchInfo bi;
    bi.n = n; bi.ref_id = "chrV"; bi.ref_pos = pos; bi.ref_base = std::string(1, ref); bi.depth = 0;
    for (uint32_t i = 0; i < n; ++i) {
        const double u = (rnd() >> 8) / 16777216.0, v = (rnd() >> 8) / 16777216.0;
        char b = 'N';
        if (u < cov) {
            b = toupper(ref) == 'N' ? 'A' : (char)toupper(ref);
            for (size_t k = 0; k < alts.size(); ++k)
                if (v >= k * alt_frac && v < (k + 1) * alt_frac) b = alts[k];
            if (v > 0.995) b = "ACGT"[rnd() % 4];   // sequencing errors
        }
        bi.align_bases.push_back(std::string(1, b));
        bi.align_base_quals.push_back((char)(33 + (b == 'N' ? 0 : 5 + rnd() % 36)));
        bi.map_strands.push_back(b == 'N' ? '.' : (rnd() & 1 ? '+' : '-'));
        bi.mapqs.push_back(b == 'N' ? 0 : (int)(rnd() % 61));
        bi.base_pos_ranks.push_back(b == 'N' ? 0 : (int)(1 + rnd() % 150));
        if (b != 'N') ++bi.depth;
    }
    return bi;
}

struct Read { char base; int phred; char strand; };
static BatchInfo make_bi(const std::string& ref, const std::vector<Read>& reads, uint32_t n) {   // padded to n samples
    BatchInfo bi;
    bi.n = n; bi.ref_id = "chrL"; bi.ref_pos = 100; bi.ref_base = ref; bi.depth = 0;
    for (uint32_t i = 0; i < n; ++i) {
        const Read r = i < reads.size() ? reads[i] : Read{'N', 0, '.'};
        bi.align_bases.push_back(std::string(1, r.base));
        bi.align_base_quals.push_back((char)(33 + r.phred));
        bi.map_strands.push_back(r.strand);
        bi.mapqs.push_back(r.base == 'N' ? 0 : 20 + (int)(i * 7 % 41));
        bi.base_pos_ranks.push_back(r.base == 'N' ? 0 : 1 + (int)(i * 13 % 150));
        if (r.base != 'N') ++bi.depth;
    }
    return bi;
}
static void add(std::vector<Read>& v, int n, char b, int q, const char* strands) {
    for (int i = 0; i < n; ++i) v.push_back(Read{b, q, strands[i % strlen(strands)]});
}

// __get_group_batchinfo: the group's samples, in sample order
static BatchInfo group_batchinfo(const BatchInfo& bi, const std::vector<size_t>& idx) {
    BatchInfo g;
    g.n = idx.size(); g.ref_id = bi.ref_id; g.ref_base = bi.ref_base; g.ref_pos = bi.ref_pos; g.depth = 0;
    for (size_t i : idx) {
        g.align_bases.push_back(bi.align_bases[i]); g.align_base_quals.push_back(bi.align_base_quals[i]);
        g.map_strands.push_back(bi.map_strands[i]); g.mapqs.push_back(bi.mapqs[i]); g.base_pos_ranks.push_back(bi.base_pos_ranks[i]);
        if (bi.align_bases[i] != "N") ++g.depth;
    }
    return g;
}

// rtol 0: bit for bit; with_qual: a group's result carries no QUAL (_out_vcf_line reads only its ALT set and AFs)
static bool same_getters(const BaseType& a, const BaseType& b, bool with_depth, bool with_qual = true, double rtol = 0) {
    auto eq = [&](double x, double y) { return rtol == 0 ? same_f64(x, y) : close_rel(x, y, rtol); };
    bool ok = a.get_alt_bases() == b.get_alt_bases() && (!with_qual || eq(a.get_var_qual(), b.get_var_qual()));
    for (char c : a.get_alt_bases()) ok = ok && eq(a.get_lrt_af(c), b.get_lrt_af(c));
    if (with_depth) {
        ok = ok && a.get_total_depth() == b.get_total_depth();
        for (char c : BASES) ok = ok && a.get_base_depth(c) == b.get_base_depth(c);
    }
    return ok;
}

static void show(const char* what, const BaseType& a, const BaseType& b) {
    static int shown = 0;
    if (++shown > 12) return;
    printf("  %s: batch", what);
    for (char c : a.get_alt_bases()) printf(" %c %.17g", c, a.get_lrt_af(c));
    printf(" qual %.17g | drop-in", a.get_var_qual());
    for (char c : b.get_alt_bases()) printf(" %c %.17g", c, b.get_lrt_af(c));
    printf(" qual %.17g\n", b.get_var_qual());
}

static int n_sites = 0, n_called = 0, n_group_checks = 0, n_group_alts = 0, n_list_checks = 0, n_last_bits = 0;

// A batch lrt(list) result (K8 or K6, lrt_on_bins) against the drop-in's BaseType(&bi, min_af).lrt(list): bit for bit.  For the
// list A,C,G,T the drop-in does not run K8 but returns the record, which K4b's thread-per-task EM decided; where several EMs
// decide the site, K4b associates its sums differently from lrt_on_bins (DESIGN.md section 8), so there the ALT set must be
// equal and AF / QUAL agree to 1e-12 relative.  Those results are counted and reported.
static bool list_matches(const BaseType& batch, const BaseType& drop, bool with_qual, bool drop_in_is_record) {
    if (same_getters(batch, drop, false, with_qual)) return true;
    if (!drop_in_is_record || !same_getters(batch, drop, false, with_qual, 1e-12)) return false;
    ++n_last_bits;
    return true;
}

// one tile through the batch path, every site against the drop-in route
static void check_tile(const char* name, const std::vector<BatchInfo>& bis, const std::map<std::string, std::vector<size_t>>& groups,
                       float min_af) {
    const uint32_t N = (uint32_t)bis[0].n, S = (uint32_t)bis.size();
    Context ctx(0, min_af, N, S, 3);
    ctx.set_groups(groups);
    // INTEGRATION.md section 2: sparse cells in, compact records out, calls and groups
    SparsePacker sp(N, S);
    TilePacker pk(N, S);
    for (const BatchInfo& bi : bis) { sp.add_site(bi); pk.add_site(bi); }
    bv_sparse_tile st = sp.tile();
    st.out_mode = BV_OUT_COMPACT;
    ctx.submit_calls(0, st);
    bv_tile dt = pk.tile();
    ctx.submit_calls(1, dt, pk.aux());               // dense records, the rpr plane from base_pos_ranks
    const TileResult r = ctx.wait_calls(0);
    const TileResult rd = ctx.wait_calls(1);
    CHECK(r.compact && !rd.compact && r.n_sites == S && r.n_groups == groups.size());
    CHECK(r.calls.size() == rd.calls.size());
    CHECK(r.calls.size() * sizeof(bv_call_out) == 0 || memcmp(r.calls.data(), rd.calls.data(), r.calls.size() * sizeof(bv_call_out)) == 0);
    CHECK(r.groups.size() * sizeof(bv_group_out) == 0 || memcmp(r.groups.data(), rd.groups.data(), r.groups.size() * sizeof(bv_group_out)) == 0);
    // [REF, ALT...] of every called site through the sparse lists path (compact: one entry per listed site)
    std::vector<uint8_t> lists((size_t)S * 4, BV_LIST_END);
    std::vector<std::vector<char>> combos(S);
    for (uint32_t i = 0; i < S; ++i) {
        const bv_site_out rec = r.record(i);
        if (!rec.n_alt) continue;
        const char up = (char)toupper(bis[i].ref_base[0]);
        combos[i].push_back(up);
        for (int k = 0; k < rec.n_alt; ++k) combos[i].push_back(BASES[rec.alt[k] & 3]);
        int n = 0;
        for (char c : combos[i]) if (code_of(c) >= 0) lists[(size_t)i * 4 + n++] = (uint8_t)code_of(c);
    }
    bv_sparse_tile lt = sp.tile();
    lt.out_mode = BV_OUT_COMPACT;
    ctx.submit_lists(2, lt, reinterpret_cast<const uint8_t(*)[4]>(lists.data()));
    const TileResult rl = ctx.wait_lists(2);
    size_t li = 0;

    std::vector<uint8_t> sample_group(N, BV_GROUP_NONE);
    uint32_t g = 0;
    for (const auto& kv : groups) { for (size_t i : kv.second) sample_group[i] = (uint8_t)g; ++g; }
    bv_params prm;
    memset(&prm, 0, sizeof(prm));
    prm.min_af = min_af; prm.lrt_threshold = 24; prm.em_max_iter = 100; prm.em_eps = 0.001f; prm.em_abs_mode = BV_EM_ABS_INT_TRUNC;

    for (uint32_t i = 0; i < S; ++i) {
        const BatchInfo& bi = bis[i];
        const bv_site_out rec = r.record(i);
        CHECK(memcmp(&rec, &rd.records[i], sizeof(rec)) == 0);   // compact sparse == dense records
        // the getters and strand_bias: batch vs drop-in
        BaseType bt(&bi, rec);
        BaseType drop(&bi, (double)min_af);
        drop.lrt();
        if (!same_getters(bt, drop, true)) { printf("FAIL %s site %u: getters differ from the drop-in route\n", name, i); ++g_fail; }
        const char up = (char)toupper(bi.ref_base[0]);
        std::string alt_string, non_ref;
        for (char c : bt.get_alt_bases()) alt_string.push_back(c);
        for (char c : BASES) if (c != up) non_ref.push_back(c);
        for (const std::string& alts : {alt_string, non_ref}) {
            if (rec.flags & BV_FLAG_BAD_STRAND) continue;
            const StrandBiasInfo a = strand_bias(up, alts, rec, &ctx), b = strand_bias(up, alts, drop.record(), &ctx);
            CHECK(a.ref_fwd == b.ref_fwd && a.ref_rev == b.ref_rev && a.alt_fwd == b.alt_fwd && a.alt_rev == b.alt_rev);
            CHECK(same_f64(a.fs, b.fs) && same_f64(a.sor, b.sor));
        }
        ++n_sites;
        const bv_call_out* call = r.call(i);
        CHECK((call != nullptr) == (rec.n_alt > 0));
        if (!call) continue;
        ++n_called;
        // the three rank sums of _out_vcf_line (src/basetype_caller.cpp:1151-1157)
        std::vector<char> first;
        for (const std::string& s : bi.align_bases) first.push_back(s[0]);
        const int mq = (int)ref_vs_alt_ranksumtest(up, alt_string, first, bi.mapqs, &ctx);
        const int rp = (int)ref_vs_alt_ranksumtest(up, alt_string, first, bi.base_pos_ranks, &ctx);
        const int bq = (int)ref_vs_alt_ranksumtest(up, alt_string, first, bi.align_base_quals, &ctx);
        if (mq != call->mq_rank_sum || rp != call->read_pos_rank_sum || bq != call->base_q_rank_sum) {
            printf("FAIL %s site %u: rank sums %d %d %d, drop-in %d %d %d\n", name, i, call->mq_rank_sum, call->read_pos_rank_sum,
                   call->base_q_rank_sum, mq, rp, bq);
            ++g_fail;
        }
        // lrt([REF, ALT...]) of the whole site: the packed list result vs the drop-in
        CHECK(li < rl.lrt.size());
        if (li < rl.lrt.size()) {
            BaseType lb(&bi, rl.lrt[li++]);
            BaseType ld(&bi, (double)min_af);
            ld.lrt(combos[i]);
            if (!list_matches(lb, ld, true, combos[i] == BASES)) {
                printf("FAIL %s site %u: lrt(list) differs from the drop-in route (flags %u)\n", name, i, rl.lrt[li - 1].flags);
                show("lrt(list)", lb, ld);
                ++g_fail;
            }
            ++n_list_checks;
        }
        // every population group: BaseType from K6's result vs BaseType(&group_bi, min_af).lrt([REF, ALT...]), and the oracle
        g = 0;
        for (const auto& kv : groups) {
            const bv_group_out* go = r.group(i, g);
            CHECK(go != nullptr);
            const BatchInfo gbi = group_batchinfo(bi, kv.second);
            BaseType gb(&bi, *go);
            BaseType gd(&gbi, (double)min_af);
            gd.lrt(combos[i]);
            if (!list_matches(gb, gd, false, combos[i] == BASES)) {
                printf("FAIL %s site %u group %s: differs from the drop-in route (flags %u)\n", name, i, kv.first.c_str(), go->flags);
                show("group", gb, gd);
                ++g_fail;
            }
            TilePacker row(N, 1, false);
            row.add_site(bi);
            const bv_tile t = row.tile();
            uint8_t order[4];
            int n_order = 0;
            for (char c : combos[i]) if (code_of(c) >= 0) order[n_order++] = (uint8_t)code_of(c);
            bv_group_out w;
            bvo_group_site(t.base, t.qual, N, sample_group.data(), g, (uint8_t)bi.ref_base[0], order, n_order, &prm, &w);
            bool ok = w.n_alt == go->n_alt;
            for (int k = 0; ok && k < w.n_alt; ++k) ok = w.alt[k] == go->alt[k] && close_rel(go->af[k], w.af[k], 1e-9);
            if (!ok) { printf("FAIL %s site %u group %s: %d ALT vs the oracle's %d\n", name, i, kv.first.c_str(), go->n_alt, w.n_alt); ++g_fail; }
            n_group_alts += go->n_alt;
            ++n_group_checks;
            ++g;
        }
    }
    CHECK(li == rl.lrt.size());
}

template <class F>
static bool throws_invalid(F f) {
    try { f(); } catch (const std::invalid_argument&) { return true; } catch (...) { return false; }
    return false;
}

int main(int argc, char** argv) {
    if (argc < 2) { printf("usage: %s <oracle library>\n", argv[0]); return 2; }
    void* h = dlopen(argv[1], RTLD_NOW);
    if (!h) { printf("dlopen %s: %s\n", argv[1], dlerror()); return 2; }
    bvo_group_site = (group_fn)dlsym(h, "bvo_group_site");
    if (!bvo_group_site) { printf("bvo_group_site not found\n"); return 2; }
    const float maf = 0.01f;

    {   // SURVEY.md 8c: G1, G2, G5, E4, E5, padded to 120 samples; three groups, some samples in none
        std::vector<Read> g1, g2, g5, e4;
        add(g1, 7, 'A', 30, "-+"); add(g1, 3, 'G', 30, "-+");
        for (int i = 0; i < 50; ++i) g2.push_back(Read{'C', 20 + i % 20, i % 3 ? '+' : '-'});
        add(g2, 5, 'T', 35, "+"); add(g2, 2, 'A', 12, "-"); add(g2, 20, 'N', 0, ".");
        add(g5, 40, 'A', 30, "-+"); add(g5, 30, 'C', 30, "-+"); add(g5, 20, 'G', 30, "+"); add(g5, 10, 'T', 30, "-");
        add(e4, 2, 'A', 30, "+"); add(e4, 2, 'C', 30, "+"); add(e4, 1, 'C', 35, "+");
        const uint32_t N = 120;
        std::vector<BatchInfo> bis = {make_bi("A", g1, N), make_bi("C", g2, N), make_bi("A", g5, N), make_bi("a", e4, N), make_bi("N", e4, N),
                                      make_bi("A", g2, N)};
        std::map<std::string, std::vector<size_t>> groups;
        for (size_t i = 0; i < N; ++i) {
            if (i % 7 == 6) continue;
            groups[i % 3 == 0 ? "EAS" : i % 3 == 1 ? "AFR" : "EUR"].push_back(i);
        }
        check_tile("SURVEY 8c", bis, groups, maf);
    }
    {   // synthetic: 400 sites x 240 samples, REF / ALT mixtures from monomorphic to tri-allelic, some lowercase / N REF
        const uint32_t N = 240, S = 400;
        std::vector<BatchInfo> bis;
        for (uint32_t s = 0; s < S; ++s) {
            const char ref = "ACGTacgN"[rnd() % 8 == 7 ? 7 : rnd() % 7];
            const uint32_t kind = rnd() % 6;
            std::string alts = kind < 2 ? "" : kind < 4 ? "G" : kind < 5 ? "TC" : "CGT";
            for (char& c : alts) if (c == toupper(ref)) c = 'A' == toupper(ref) ? 'C' : 'A';
            bis.push_back(make_site(N, ref, alts, 0.05 + (rnd() % 90) / 100.0, 0.02 + (rnd() % 20) / 100.0, 1000 + s));
        }
        std::map<std::string, std::vector<size_t>> groups;
        for (size_t i = 0; i < N; ++i) {
            const uint32_t u = rnd() % 5;
            if (u < 4) groups[std::string("pop") + (char)('A' + u)].push_back(i);
        }
        check_tile("synthetic", bis, groups, maf);
    }
    {   // set_groups refusals
        Context ctx(0, maf, 10, 4, 1);
        std::map<std::string, std::vector<size_t>> twice = {{"a", {0, 1}}, {"b", {1, 2}}};
        CHECK(throws_invalid([&] { ctx.set_groups(twice); }));
        std::map<std::string, std::vector<size_t>> out_of_range = {{"a", {0, 10}}};
        CHECK(throws_invalid([&] { ctx.set_groups(out_of_range); }));
        std::map<std::string, std::vector<size_t>> many;
        for (int k = 0; k <= BV_MAX_GROUPS; ++k) many["g" + std::to_string(1000 + k)] = {};
        CHECK(throws_invalid([&] { ctx.set_groups(many); }));
        CHECK(ctx.n_groups() == 0);
    }
    printf("%d sites, %d called, %d lists, %d group results (%d group ALT alleles) checked against the drop-in route; "
           "%d list / group results of the list A,C,G,T equal to the record to 1e-12 but not bit for bit\n", n_sites, n_called, n_list_checks, n_group_checks, n_group_alts,
           n_last_bits);
    CHECK(n_called > 50 && n_group_alts > 50);
    if (g_fail) { printf("%d FAILURES\n", g_fail); return 1; }
    printf("ALL OK\n");
    return 0;
}
