// GPU test of BaseType(&bi, min_af).lrt(list) in the C++ host mirror: the known-answer vectors of SURVEY.md 8c (G1, G2, G5,
// E4, E5) with reordered and shortened candidate lists against the oracle's bvo_site_list on the same rows, the mono-allelic
// QUAL rule reached through a list whose first active base is not REF, and the refusals (repeated base, record-built object).
// TEST INFRASTRUCTURE: loads the list oracle (tests/oracle_lists.c, built by tests/oracle_lists.py; its path is the first
// argument) through dlopen; the host library itself never touches it.
#include <dlfcn.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../basevar_b200/host/bv_host.hpp"

using namespace bvhost;

static int g_fail = 0;
#define CHECK(cond)                                                        \
    do {                                                                   \
        if (!(cond)) { printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); ++g_fail; } \
    } while (0)

typedef int (*list_fn)(const uint8_t*, const uint8_t*, const uint8_t*, uint32_t, uint8_t, const uint8_t*, int, const bv_params*,
                       bv_lrt_out*);
static list_fn bvo_site_list = nullptr;

static bool close_rel(double a, double b, double rtol = 1e-9, double atol = 1e-12) {
    if (std::isnan(a) && std::isnan(b)) return true;
    return a == b || std::fabs(a - b) <= atol + rtol * std::fabs(b);
}

struct Read { char base; int phred; char strand; };

static BatchInfo make_bi(const std::string& ref, const std::vector<Read>& reads) {
    BatchInfo bi;
    bi.n = reads.size(); bi.ref_id = "chrL"; bi.ref_pos = 100; bi.ref_base = ref; bi.depth = 0;
    for (const Read& r : reads) {
        bi.align_bases.push_back(std::string(1, r.base));
        bi.align_base_quals.push_back((char)(33 + r.phred));
        bi.map_strands.push_back(r.strand);
        bi.mapqs.push_back(60); bi.base_pos_ranks.push_back(1);
        if (r.base != 'N') ++bi.depth;
    }
    return bi;
}

static void add(std::vector<Read>& v, int n, char b, int q, const char* strands) {   // strands cycle through the string
    for (int i = 0; i < n; ++i) v.push_back(Read{b, q, strands[i % strlen(strands)]});
}

// the oracle on the same row: BatchInfo -> encoded planes (TilePacker, pageable) -> bvo_site_list
static bv_lrt_out oracle(const BatchInfo& bi, float min_af, const std::vector<char>& list) {
    TilePacker pk((uint32_t)bi.n, 1, false);
    pk.add_site(bi);
    const bv_tile t = pk.tile();
    uint8_t codes[4];
    int n = 0;
    for (char c : list) {
        const int k = c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1;
        if (k >= 0) codes[n++] = (uint8_t)k;
    }
    bv_params p;
    memset(&p, 0, sizeof(p));
    p.min_af = min_af; p.lrt_threshold = 24; p.em_max_iter = 100; p.em_eps = 0.001f; p.em_abs_mode = BV_EM_ABS_INT_TRUNC;
    bv_lrt_out o;
    CHECK(bvo_site_list(t.base, t.qual, t.strand, (uint32_t)bi.n, t.ref_base[0], codes, n, &p, &o) == 0);
    return o;
}

static int n_checked = 0, n_mono = 0;

static void check_list(const char* name, const BatchInfo& bi, const std::vector<char>& list) {
    const float maf = 0.01f;
    BaseType bt(&bi, (double)maf);
    bt.lrt(list);
    const bv_lrt_out w = oracle(bi, maf, list);
    const std::vector<char>& alts = bt.get_alt_bases();
    bool ok = alts.size() == w.n_alt;
    for (size_t k = 0; ok && k < alts.size(); ++k) {
        ok = alts[k] == BASES[w.alt[k]] && close_rel(bt.get_lrt_af(alts[k]), w.af[k]);
    }
    ok = ok && close_rel(bt.get_var_qual(), w.qual);
    if (!ok) {
        std::string l(list.begin(), list.end());
        printf("FAIL %s lrt({%s}): %zu ALT, qual %.17g; oracle %d ALT, qual %.17g\n", name, l.c_str(), alts.size(), bt.get_var_qual(),
               (int)w.n_alt, w.qual);
        ++g_fail;
    }
    if (w.flags & BV_FLAG_MONO_QUAL) { ++n_mono; CHECK(bt.get_var_qual() == 5000.0); }
    ++n_checked;
}

int main(int argc, char** argv) {
    if (argc < 2) { printf("FAIL usage: test_lists_gpu <path of the list oracle library>\n"); return 1; }
    void* ho = dlopen(argv[1], RTLD_NOW);
    if (!ho) { printf("FAIL cannot load the oracle: %s\n", dlerror()); return 1; }
    bvo_site_list = (list_fn)dlsym(ho, "bvo_site_list");
    if (!bvo_site_list) { printf("FAIL bvo_site_list missing\n"); return 1; }

    // SURVEY.md 8c
    std::vector<Read> g1, g2, g5, e4;
    add(g1, 7, 'A', 30, "-+"); add(g1, 3, 'G', 30, "-+");
    for (int i = 0; i < 50; ++i) g2.push_back(Read{'C', 20 + i % 20, i % 3 ? '+' : '-'});
    add(g2, 5, 'T', 35, "+"); add(g2, 2, 'A', 12, "-"); add(g2, 20, 'N', 0, ".");
    add(g5, 40, 'A', 30, "-+"); add(g5, 30, 'C', 30, "-+"); add(g5, 20, 'G', 30, "+"); add(g5, 10, 'T', 30, "-");
    add(e4, 2, 'A', 30, "+"); add(e4, 2, 'C', 30, "+"); add(e4, 1, 'C', 35, "+");
    struct Vec { const char* name; BatchInfo bi; };
    std::vector<Vec> vecs = {{"G1", make_bi("A", g1)}, {"G2", make_bi("C", g2)}, {"G5", make_bi("A", g5)}, {"E4", make_bi("a", e4)},
                             {"E5", make_bi("N", e4)},
                             // G2's reads under REF A: lrt({C}) reaches the mono-allelic rule through a base that is not REF
                             {"G2/refA", make_bi("A", g2)}};
    const std::vector<std::vector<char>> lists = {
        {'A', 'C', 'G', 'T'}, {'T', 'G', 'C', 'A'}, {'G', 'A'}, {'A', 'G'}, {'C', 'T'}, {'T', 'C', 'A'}, {'C'}, {'G'}, {'A'},
        {'C', 'A', 'G'}, {'G', 'T', 'C'}, {'C', 'N', 'A'}, {'a', 'C'}, {'T', 'A', 'C', 'G'}, {'N'}, {}};
    for (const Vec& v : vecs)
        for (const auto& l : lists) check_list(v.name, v.bi, l);
    {   // the known answer of G1 (SURVEY.md 8c) through a reordered list
        BaseType bt(&vecs[0].bi, (double)0.01f);
        bt.lrt({'G', 'A'});
        CHECK(bt.get_alt_bases().size() == 1 && bt.get_alt_bases()[0] == 'G');
        CHECK(close_rel(bt.get_lrt_af('G'), 0.2998664889880594) && close_rel(bt.get_var_qual(), 86.650670492227547));
    }
    {   // G5 with the list in reverse: ALT in list order T, G, C (the reference's own ALT order follows the list)
        BaseType bt(&vecs[2].bi, (double)0.01f);
        bt.lrt({'T', 'G', 'C', 'A'});
        CHECK(bt.get_alt_bases() == std::vector<char>({'T', 'G', 'C'}));
        CHECK(close_rel(bt.get_lrt_af('C'), 0.30006675422865065) && close_rel(bt.get_var_qual(), 217.57830376056739));
    }
    {   // mono-allelic rule: one active base, not REF, total 57 > 10, 50/57 > 0.5
        BaseType bt(&vecs[5].bi, (double)0.01f);
        bt.lrt({'C'});
        CHECK(bt.get_alt_bases() == std::vector<char>({'C'}) && bt.get_var_qual() == 5000.0);
    }
    {   // refusals
        BaseType bt(&vecs[0].bi, (double)0.01f);
        bool threw = false;
        try { bt.lrt({'A', 'G', 'A'}); } catch (const std::invalid_argument&) { threw = true; }
        CHECK(threw);
        bv_site_out r;
        memset(&r, 0, sizeof(r));
        BaseType from_rec(&vecs[0].bi, r);
        threw = false;
        try { from_rec.lrt({'A', 'G'}); } catch (const std::invalid_argument&) { threw = true; }
        CHECK(threw);
    }
    CHECK(n_mono >= 1);
    printf("%d lists checked against the oracle, %d through the mono-allelic rule\n", n_checked, n_mono);
    if (g_fail) { printf("%d FAILURES\n", g_fail); return 1; }
    printf("ALL OK\n");
    return 0;
}
