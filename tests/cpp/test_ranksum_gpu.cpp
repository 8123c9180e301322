// GPU test of ref_vs_alt_ranksumtest in the C++ host mirror (both overloads): the known-answer vector of SURVEY.md 8c against
// the oracle's bvo_wilcoxon, skipped N / indel bases, chars at or above 128 in the char overload, every std::invalid_argument
// case, and the three values of a called site, truncated, against the batch path's bv_call_out.
// TEST INFRASTRUCTURE: loads the oracle library (oracle/libbvoracle.so; its path is the first argument) through dlopen; the
// host library itself never touches it.
#include <dlfcn.h>

#include <cmath>
#include <cstdio>
#include <cstring>
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

typedef double (*wilcoxon_fn)(const double*, size_t, const double*, size_t);
static wilcoxon_fn bvo_wilcoxon = nullptr;

static bool close_rel(double a, double b) { return a == b || std::fabs(a - b) <= 1e-12 + 1e-9 * std::fabs(b); }

// the oracle's answer for explicit classes: -10 log10 of bvo_wilcoxon, 10000 for an empty class or p == 0
static double oracle(const std::vector<double>& r, const std::vector<double>& a) {
    if (r.empty() || a.empty()) return 10000;
    double v = -10 * log10(bvo_wilcoxon(r.data(), r.size(), a.data(), a.size()));
    return std::isinf(v) ? 10000 : v;
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
    bvo_wilcoxon = (wilcoxon_fn)dlsym(h, "bvo_wilcoxon");
    if (!bvo_wilcoxon) { printf("bvo_wilcoxon not found\n"); return 2; }

    // SURVEY.md 8c: wilcoxon_ranksum_test({1,5,3,10,3,3,4,5},{6,7,2,2,8,9,10}) -> 0.271589; here REF A, ALT C
    const std::vector<double> s1 = {1, 5, 3, 10, 3, 3, 4, 5}, s2 = {6, 7, 2, 2, 8, 9, 10};
    std::vector<char> bases;
    std::vector<int> vi;
    std::vector<char> vc;
    for (double x : s1) { bases.push_back('A'); vi.push_back((int)x); vc.push_back((char)x); }
    for (double x : s2) { bases.push_back('C'); vi.push_back((int)x); vc.push_back((char)x); }
    const double want = oracle(s1, s2);
    CHECK(std::fabs(std::pow(10.0, -want / 10) - 0.271589) < 5e-7);
    const double got_i = ref_vs_alt_ranksumtest('A', "C", bases, vi);
    const double got_c = ref_vs_alt_ranksumtest('A', "C", bases, vc);
    CHECK(close_rel(got_i, want));
    CHECK(close_rel(got_c, want));
    printf("known answer: %.9f (oracle %.9f), p = %.6f\n", got_i, want, std::pow(10.0, -got_i / 10));
    // an ALT set that holds REF changes nothing; REF N puts A/C/G/T reads in the ALT class or in neither
    CHECK(ref_vs_alt_ranksumtest('A', "AC", bases, vi) == got_i);
    CHECK(ref_vs_alt_ranksumtest('N', "C", bases, vi) == 10000);

    // N, insertions, deletions and other characters are in neither class
    {
        std::vector<char> b2 = bases;
        std::vector<int> v2 = vi;
        const char extra[] = {'N', '+', '-', '*', 'N'};
        for (char c : extra) { b2.push_back(c); v2.push_back(1000); }
        CHECK(ref_vs_alt_ranksumtest('A', "C", b2, v2) == got_i);
    }

    // chars at or above 128 widen as signed chars: values -128..-1 rank below every value 0..127
    {
        std::vector<char> b3, v3;
        std::vector<double> r, a;
        for (int i = 0; i < 40; ++i) {
            const unsigned char u = (unsigned char)(i * 37 % 256);
            const bool is_ref = i % 3 != 0;
            b3.push_back(is_ref ? 'G' : 'T');
            v3.push_back((char)u);
            (is_ref ? r : a).push_back((double)(signed char)u);
        }
        const double g = ref_vs_alt_ranksumtest('G', "T", b3, v3);
        CHECK(close_rel(g, oracle(r, a)));
        printf("signed chars: %.9f (oracle %.9f)\n", g, oracle(r, a));
    }

    // all tied: -0.0; one class empty: 10000
    {
        std::vector<int> tied(bases.size(), 30);
        const double t = ref_vs_alt_ranksumtest('A', "C", bases, tied);
        CHECK(t == 0.0 && std::signbit(t));
        CHECK(ref_vs_alt_ranksumtest('A', "G", bases, vi) == 10000);
        CHECK(ref_vs_alt_ranksumtest('A', "C", std::vector<char>(), std::vector<int>()) == 10000);
    }

    // std::invalid_argument: sizes differ; an ALT character that is not A/C/G/T; a lowercase REF; a REF other than A/C/G/T/N
    // that some base equals
    CHECK(throws_invalid([&] { ref_vs_alt_ranksumtest('A', "C", bases, std::vector<int>(3, 1)); }));
    CHECK(throws_invalid([&] { ref_vs_alt_ranksumtest('A', "C", bases, std::vector<char>(3, 1)); }));
    CHECK(throws_invalid([&] { ref_vs_alt_ranksumtest('A', "CN", bases, vi); }));
    CHECK(throws_invalid([&] { ref_vs_alt_ranksumtest('A', "c", bases, vi); }));
    CHECK(throws_invalid([&] { ref_vs_alt_ranksumtest('a', "C", bases, vi); }));
    {
        std::vector<char> b4 = bases;
        std::vector<int> v4 = vi;
        b4.push_back('*'); v4.push_back(3);
        CHECK(throws_invalid([&] { ref_vs_alt_ranksumtest('*', "C", b4, v4); }));
        CHECK(ref_vs_alt_ranksumtest('*', "C", bases, vi) == 10000);   // no base equals it: no REF read
    }
    printf("refusals checked\n");

    // a called site through the batch path (bv_tile_submit_calls) and through the mirror: MQRankSum, ReadPosRankSum and
    // BaseQRankSum as _out_vcf_line forms them (src/basetype_caller.cpp:1151-1157)
    {
        const uint32_t N = 600;
        BatchInfo bi;
        bi.n = N; bi.ref_id = "chrR"; bi.ref_pos = 7; bi.ref_base = "G"; bi.depth = 0;
        uint32_t x = 12345;
        auto rnd = [&]() { x = x * 1103515245u + 12345u; return (x >> 8) & 0xffffu; };
        for (uint32_t i = 0; i < N; ++i) {
            const uint32_t u = rnd() % 100;
            const char b = u < 55 ? 'G' : u < 85 ? 'A' : u < 88 ? 'T' : u < 92 ? 'N' : u < 95 ? 'C' : u < 97 ? '+' : '-';
            bi.align_bases.push_back(b == '+' ? std::string("+AC") : b == '-' ? std::string("-T") : std::string(1, b));
            bi.align_base_quals.push_back((char)(33 + 5 + rnd() % 36));
            bi.map_strands.push_back(rnd() & 1 ? '+' : '-');
            bi.mapqs.push_back((int)(rnd() % 61));
            bi.base_pos_ranks.push_back((int)(1 + rnd() % 150));
        }
        TilePacker pk(N, 1);
        pk.add_site(bi);
        const bv_tile t = pk.tile();
        std::vector<uint16_t> rpr((N + 7) / 8 * 8, 0);
        for (uint32_t i = 0; i < N; ++i) rpr[i] = (uint16_t)bi.base_pos_ranks[i];
        bv_tile_aux aux;
        aux.mapq = pk.mapq_plane(); aux.rpr = rpr.data(); aux.rpr_pitch = rpr.size();
        Context ctx(0, 0.01f, N, 1, 1);
        CHECK(bv_tile_submit_calls(ctx.raw(), 0, &t, &aux) == BV_OK);
        bv_site_out rec;
        bv_call_out call;
        uint32_t n_calls = 0;
        CHECK(bv_tile_wait_calls(ctx.raw(), 0, &rec, &call, 1, &n_calls, nullptr) == BV_OK);
        CHECK(n_calls == 1 && rec.n_alt > 0);
        if (n_calls == 1) {
            std::string alts;
            for (int k = 0; k < rec.n_alt; ++k) alts.push_back(BASES[rec.alt[k] & 3]);
            std::vector<char> first;   // the first character of each align_base, as the reference's caller passes them
            for (const std::string& s : bi.align_bases) first.push_back(s[0]);
            const int mq = (int)ref_vs_alt_ranksumtest('G', alts, first, bi.mapqs);
            const int rp = (int)ref_vs_alt_ranksumtest('G', alts, first, bi.base_pos_ranks);
            const int bq = (int)ref_vs_alt_ranksumtest('G', alts, first, bi.align_base_quals, &ctx);
            CHECK(mq == call.mq_rank_sum);
            CHECK(rp == call.read_pos_rank_sum);
            CHECK(bq == call.base_q_rank_sum);
            printf("called site ALT %s: mirror %d %d %d, bv_call_out %d %d %d\n", alts.c_str(), mq, rp, bq, call.mq_rank_sum,
                   call.read_pos_rank_sum, call.base_q_rank_sum);
        }
    }

    if (g_fail) { printf("%d FAILURES\n", g_fail); return 1; }
    printf("ALL OK\n");
    return 0;
}
