// GPU test of Context::run_device in the C++ host mirror: the SURVEY.md 8c vectors and a synthetic tile, packed with SparsePacker
// and TilePacker, copied to device memory and run there (sparse cells and dense planes; records and compact results; plain,
// called sites and lists), against Context::submit / wait of the same host tiles: the results must be the same bytes (compact
// records compared through their briefs, called sites by row).
// TEST INFRASTRUCTURE: the device buffers are allocated with the CUDA runtime here; the host library itself never touches
// device memory.
#include <cuda_runtime.h>

#include <algorithm>
#include <cctype>
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

static uint32_t g_x = 88172645u;
static uint32_t rnd() { g_x ^= g_x << 13; g_x ^= g_x >> 17; g_x ^= g_x << 5; return g_x; }

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
static BatchInfo make_site(uint32_t n, char ref, const std::string& alts, double cov, double alt_frac) {
    std::vector<Read> reads;
    for (uint32_t i = 0; i < n; ++i) {
        const double u = (rnd() >> 8) / 16777216.0, v = (rnd() >> 8) / 16777216.0;
        char b = 'N';
        if (u < cov) {
            b = toupper(ref) == 'N' ? 'A' : (char)toupper(ref);
            for (size_t k = 0; k < alts.size(); ++k)
                if (v >= k * alt_frac && v < (k + 1) * alt_frac) b = alts[k];
        }
        reads.push_back(b == 'N' ? Read{'N', 0, '.'} : Read{b, 5 + (int)(rnd() % 36), (rnd() & 1) ? '+' : '-'});
    }
    return make_bi(std::string(1, ref), reads, n);
}

// device copy of a host array (freed at exit of the test by the runtime)
template <class T>
static T* to_device(const T* p, size_t n) {
    void* d = nullptr;
    if (cudaMalloc(&d, std::max<size_t>(n * sizeof(T), 16)) != cudaSuccess) { printf("cudaMalloc failed\n"); exit(2); }
    if (n) cudaMemcpy(d, p, n * sizeof(T), cudaMemcpyHostToDevice);
    return static_cast<T*>(d);
}
template <class T>
static T* device_buffer(size_t n) {
    void* d = nullptr;
    if (cudaMalloc(&d, std::max<size_t>(n * sizeof(T), 16)) != cudaSuccess) { printf("cudaMalloc failed\n"); exit(2); }
    cudaMemset(d, 0xee, std::max<size_t>(n * sizeof(T), 16));
    return static_cast<T*>(d);
}
template <class T>
static std::vector<T> to_host(const T* d, size_t n) {
    std::vector<T> v(n);
    if (n) cudaMemcpy(v.data(), d, n * sizeof(T), cudaMemcpyDeviceToHost);
    return v;
}
static uint32_t word(const uint32_t* d) { return to_host(d, 1)[0]; }

// records of a compact result: full record where the brief points, else bv_site_expand
static std::vector<bv_site_out> expand(const std::vector<bv_site_brief>& b, const bv_site_out* full, uint32_t n_full, const uint8_t* ref, float maf) {
    std::vector<bv_site_out> out(b.size());
    for (size_t i = 0; i < b.size(); ++i) {
        if (b[i].w0 & 0x80000000u) {
            const uint32_t k = b[i].w0 & 0x7fffffffu;
            if (k < n_full) out[i] = full[k];
            else { ++g_fail; printf("FAIL: brief %zu points past the full records\n", i); }
        } else {
            bv_site_expand(&b[i], ref[i], maf, &out[i]);
        }
    }
    return out;
}
static bool same_records(const std::vector<bv_site_out>& a, const std::vector<bv_site_out>& b) {
    return a.size() == b.size() && (a.empty() || memcmp(a.data(), b.data(), a.size() * sizeof(bv_site_out)) == 0);
}
static std::vector<bv_call_out> by_site(std::vector<bv_call_out> c) {
    std::sort(c.begin(), c.end(), [](const bv_call_out& x, const bv_call_out& y) { return x.site < y.site; });
    return c;
}

static int n_checked = 0;

static void check_tile(const char* name, const std::vector<BatchInfo>& bis, float maf) {
    const uint32_t S = (uint32_t)bis.size(), N = (uint32_t)bis[0].n;
    Context ctx(0, maf, N, S, 1);
    SparsePacker sp(N, S);
    TilePacker tp(N, S);
    for (const BatchInfo& bi : bis) { sp.add_site(bi); tp.add_site(bi); }
    const bv_sparse_tile ht = sp.tile();
    const uint64_t n_cells = ht.site_start[S];
    std::vector<uint8_t> ref(ht.ref_base, ht.ref_base + S);
    // the same cells in device memory
    bv_sparse_tile dt = ht;
    dt.cells = to_device(static_cast<const uint32_t*>(ht.cells), n_cells);
    dt.cells_aux = to_device(ht.cells_aux, n_cells);
    dt.site_start = to_device(ht.site_start, S + 1);
    dt.ref_base = to_device(ht.ref_base, S);
    dt.out = nullptr;
    // lists: [REF?, A, C, G, T] in a rotating order, some empty
    std::vector<uint8_t> lists((size_t)S * 4, BV_LIST_END);
    for (uint32_t i = 0; i < S; ++i)
        for (uint32_t k = 0; k < i % 5; ++k) lists[(size_t)i * 4 + k] = (uint8_t)((i + k) % 4);
    const uint8_t(*hl)[4] = reinterpret_cast<const uint8_t(*)[4]>(lists.data());
    const uint8_t(*dl)[4] = reinterpret_cast<const uint8_t(*)[4]>(to_device(lists.data(), lists.size()));

    bv_site_out* d_out = device_buffer<bv_site_out>(S);
    bv_site_brief* d_brief = device_buffer<bv_site_brief>(S);
    bv_site_out* d_full = device_buffer<bv_site_out>(S);
    bv_call_out* d_calls = device_buffer<bv_call_out>(S);
    bv_lrt_out* d_lrt = device_buffer<bv_lrt_out>(S);
    uint32_t* d_words = device_buffer<uint32_t>(4);   // n_full, n_calls, n_lrt, status

    for (int compact = 0; compact < 2; ++compact) {
        const int mode = compact ? BV_OUT_COMPACT : BV_OUT_RECORDS;
        for (int kind : {BV_RUN_PLAIN, BV_RUN_CALLS, BV_RUN_LISTS}) {
            // host route
            bv_sparse_tile h = ht;
            h.out_mode = (uint32_t)mode;
            TileResult want;
            if (kind == BV_RUN_PLAIN) {
                ctx.submit(0, h);
                if (compact) {
                    const bv_site_brief* b; const bv_site_out* f; uint32_t nf;
                    CHECK(bv_tile_wait_compact(ctx.raw(), 0, &b, &f, &nf) == BV_OK);
                    want.records = expand(std::vector<bv_site_brief>(b, b + S), f, nf, ref.data(), maf);
                } else {
                    want.records.resize(S);
                    ctx.wait(0, want.records.data());
                }
            } else if (kind == BV_RUN_CALLS) {
                ctx.submit_calls(0, h);
                want = ctx.wait_calls(0);
            } else {
                ctx.submit_lists(0, h, hl);
                want = ctx.wait_lists(0);
            }
            std::vector<bv_site_out> want_rec(S);
            for (uint32_t i = 0; i < S; ++i) want_rec[i] = kind == BV_RUN_PLAIN ? want.records[i] : want.record(i);
            // device route
            DeviceResult o(kind, mode);
            o.d_out = d_out; o.d_brief = d_brief; o.d_full = d_full; o.d_n_full = d_words;
            o.d_calls = d_calls; o.d_n_calls = d_words + 1;
            o.d_lists = dl; o.d_lrt = d_lrt; o.d_n_lrt = d_words + 2;
            o.d_status = d_words + 3;
            ctx.run_device(dt, o);
            cudaDeviceSynchronize();
            CHECK(word(d_words + 3) == 0);
            std::vector<bv_site_out> got_rec;
            if (compact) {
                const uint32_t nf = word(d_words);
                const std::vector<bv_site_out> full = to_host(d_full, nf);
                got_rec = expand(to_host(d_brief, S), full.data(), nf, ref.data(), maf);
            } else {
                got_rec = to_host(d_out, S);
            }
            if (!same_records(got_rec, want_rec)) { printf("FAIL %s kind %d compact %d: records differ\n", name, kind, compact); ++g_fail; }
            if (kind == BV_RUN_CALLS) {
                const std::vector<bv_call_out> got = by_site(to_host(d_calls, word(d_words + 1))), exp = by_site(want.calls);
                CHECK(got.size() == exp.size() && (got.empty() || memcmp(got.data(), exp.data(), got.size() * sizeof(bv_call_out)) == 0));
            }
            if (kind == BV_RUN_LISTS) {
                const size_t n = compact ? word(d_words + 2) : S;
                const std::vector<bv_lrt_out> got = to_host(d_lrt, n);
                CHECK(got.size() == want.lrt.size() && (got.empty() || memcmp(got.data(), want.lrt.data(), n * sizeof(bv_lrt_out)) == 0));
            }
            ++n_checked;
        }
    }
    // dense planes in device memory (bv_tile_run_device_ex) against the host dense tile
    const bv_tile hd = tp.tile();
    const std::vector<bv_site_out> want = ctx.run(hd);
    bv_tile dd = hd;
    const size_t plane = (size_t)S * hd.pitch;
    dd.base = to_device(hd.base, plane); dd.qual = to_device(hd.qual, plane); dd.strand = to_device(hd.strand, plane);
    dd.ref_base = to_device(hd.ref_base, S);
    dd.location = BV_LOC_DEVICE;
    for (int compact = 0; compact < 2; ++compact) {
        DeviceResult o(BV_RUN_PLAIN, compact ? BV_OUT_COMPACT : BV_OUT_RECORDS);
        o.d_out = d_out; o.d_brief = d_brief; o.d_full = d_full; o.d_n_full = d_words;
        ctx.run_device(dd, o);
        cudaDeviceSynchronize();
        const std::vector<bv_site_out> got = compact ? expand(to_host(d_brief, S), to_host(d_full, word(d_words)).data(), word(d_words), ref.data(), maf)
                                                     : to_host(d_out, S);
        if (!same_records(got, want)) { printf("FAIL %s dense compact %d: records differ\n", name, compact); ++g_fail; }
        ++n_checked;
    }
    // host memory is refused, nothing queued
    bool threw = false;
    try {
        DeviceResult o(BV_RUN_PLAIN, BV_OUT_RECORDS);
        o.d_out = d_out;
        ctx.run_device(ht, o);
    } catch (const std::runtime_error&) { threw = true; }
    CHECK(threw);
}

int main() {
    const float maf = 0.01f;
    {   // SURVEY.md 8c: G1, G2, G5, E4 (lowercase and N REF), padded to 120 samples
        std::vector<Read> g1, g2, g5, e4;
        add(g1, 7, 'A', 30, "-+"); add(g1, 3, 'G', 30, "-+");
        for (int i = 0; i < 50; ++i) g2.push_back(Read{'C', 20 + i % 20, i % 3 ? '+' : '-'});
        add(g2, 5, 'T', 35, "+"); add(g2, 2, 'A', 12, "-"); add(g2, 20, 'N', 0, ".");
        add(g5, 40, 'A', 30, "-+"); add(g5, 30, 'C', 30, "-+"); add(g5, 20, 'G', 30, "+"); add(g5, 10, 'T', 30, "-");
        add(e4, 2, 'A', 30, "+"); add(e4, 2, 'C', 30, "+"); add(e4, 1, 'C', 35, "+");
        const uint32_t N = 120;
        check_tile("SURVEY 8c", {make_bi("A", g1, N), make_bi("C", g2, N), make_bi("A", g5, N), make_bi("a", e4, N), make_bi("N", e4, N),
                                 make_bi("A", g2, N)}, maf);
    }
    {   // synthetic: 700 sites x 300 samples, monomorphic to tri-allelic, some lowercase / N REF
        const uint32_t N = 300, S = 700;
        std::vector<BatchInfo> bis;
        for (uint32_t s = 0; s < S; ++s) {
            const char ref = "ACGTacgN"[rnd() % 8];
            const uint32_t kind = rnd() % 6;
            std::string alts = kind < 3 ? "" : kind < 4 ? "G" : kind < 5 ? "TC" : "CGT";
            for (char& c : alts) if (c == toupper(ref)) c = 'A' == toupper(ref) ? 'C' : 'A';
            bis.push_back(make_site(N, ref, alts, 0.02 + (rnd() % 90) / 100.0, 0.02 + (rnd() % 20) / 100.0));
        }
        check_tile("synthetic", bis, maf);
    }
    printf("%d device-resident results checked against the host route\n", n_checked);
    if (g_fail) { printf("%d FAILURES\n", g_fail); return 1; }
    printf("ALL OK\n");
    return 0;
}
