// bv_host.cpp -- see bv_host.hpp.  Host-side plumbing only: packing, contexts, record -> BaseType, region sharding.
#include "bv_host.hpp"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <mutex>
#include <thread>

namespace bvhost {

static void check(int rc, bv_ctx* ctx, const char* what) {
    if (rc != BV_OK) throw std::runtime_error(std::string("[ERROR] ") + what + ": " + bv_last_error(ctx));
}

uint8_t encode_base(const std::string& s) {
    const char fb = s.empty() ? 'N' : s[0];
    if (fb == 'N') return BV_BASE_N;
    if (fb == '+') return BV_BASE_INS;
    if (fb == '-') return BV_BASE_DEL;
    if (s.size() != 1)   // src/basetype.cpp:54-56
        throw std::runtime_error("[ERROR] Why dose the size of aligned base is not 1? Check: " + s);
    switch (fb) {
        case 'A': return BV_BASE_A;
        case 'C': return BV_BASE_C;
        case 'G': return BV_BASE_G;
        case 'T': return BV_BASE_T;
        default: return BV_BASE_OTHER;   // counted in the total depth, never an allele (src/basetype.cpp:58-64)
    }
}

float cli_min_af(float min_af, size_t n_bam) { return std::min(float(100) / n_bam, min_af); }

// ---- TilePacker ------------------------------------------------------------------------------------------------------
static uint8_t* plane_alloc(size_t bytes, bool pinned) {
    void* p = nullptr;
    if (pinned) {
        if (bv_host_alloc(&p, bytes) != BV_OK) throw std::runtime_error(std::string("[ERROR] bv_host_alloc: ") + bv_last_error(nullptr));
    } else {
        if (posix_memalign(&p, 64, bytes ? bytes : 64) != 0) throw std::bad_alloc();
    }
    return static_cast<uint8_t*>(p);
}
static void plane_free(uint8_t* p, bool pinned) {
    if (!p) return;
    if (pinned) bv_host_free(p);
    else free(p);
}

TilePacker::TilePacker(uint32_t n_samples, uint32_t max_sites, bool pinned)
    : n_samples_(n_samples), max_sites_(max_sites), pitch_(((uint64_t)n_samples + 15) / 16 * 16), pinned_(pinned) {
    const size_t plane = (size_t)max_sites_ * pitch_;
    base_ = plane_alloc(plane, pinned_);
    qual_ = plane_alloc(plane, pinned_);
    strand_ = plane_alloc(plane, pinned_);
    mapq_ = plane_alloc(plane, pinned_);
    rpr_ = reinterpret_cast<uint16_t*>(plane_alloc(plane * sizeof(uint16_t), pinned_));
    ref_ = plane_alloc(max_sites_, pinned_);
}

TilePacker::~TilePacker() {
    plane_free(base_, pinned_); plane_free(qual_, pinned_); plane_free(strand_, pinned_); plane_free(mapq_, pinned_);
    plane_free(reinterpret_cast<uint8_t*>(rpr_), pinned_); plane_free(ref_, pinned_);
}

void TilePacker::next_row(char ref_base, uint8_t** b, uint8_t** q, uint8_t** s, uint8_t** m) {
    if (n_sites_ >= max_sites_) throw std::runtime_error("[ERROR] TilePacker is full");
    const size_t row = (size_t)n_sites_ * pitch_;
    // uncovered = N ! 0 0 . (src/basetype_caller.cpp:1051-1077)
    memset(base_ + row, BV_BASE_N, pitch_);
    memset(qual_ + row, 0, pitch_);
    memset(strand_ + row, BV_STRAND_NONE, pitch_);
    memset(mapq_ + row, 0, pitch_);
    memset(rpr_ + row, 0, pitch_ * sizeof(uint16_t));
    ref_[n_sites_] = (uint8_t)ref_base;
    *b = base_ + row; *q = qual_ + row; *s = strand_ + row; *m = mapq_ + row;
    ++n_sites_;
}

void TilePacker::add_site_cells(char ref_base, const uint8_t* base, const uint8_t* qual, const uint8_t* strand, const uint8_t* mapq) {
    uint8_t *b, *q, *s, *m;
    next_row(ref_base, &b, &q, &s, &m);
    memcpy(b, base, n_samples_); memcpy(q, qual, n_samples_); memcpy(s, strand, n_samples_);
    if (mapq) memcpy(m, mapq, n_samples_);
}

bv_tile TilePacker::tile() const {
    bv_tile t;
    t.base = base_; t.qual = qual_; t.strand = strand_; t.ref_base = ref_;
    t.pitch = pitch_; t.n_sites = n_sites_; t.n_samples = n_samples_;
    t.location = BV_LOC_HOST; t.out_mode = BV_OUT_RECORDS;
    return t;
}

bv_tile_aux TilePacker::aux() const {
    bv_tile_aux a;
    a.mapq = mapq_; a.rpr = rpr_; a.rpr_pitch = pitch_;
    return a;
}

// ---- SparsePacker -----------------------------------------------------------------------------------------------------
SparsePacker::SparsePacker(uint32_t n_samples, uint32_t max_sites, size_t reserve_cells) : n_samples_(n_samples), max_sites_(max_sites) {
    if (n_samples > BV_CELL_MAX_SAMPLES) throw std::runtime_error("[ERROR] sparse tiles hold at most 2^20 samples");
    site_start_ = reinterpret_cast<uint32_t*>(plane_alloc(((size_t)max_sites + 1) * sizeof(uint32_t), true));
    ref_ = plane_alloc(max_sites ? max_sites : 1, true);
    site_start_[0] = 0;
    grow(reserve_cells ? reserve_cells : (size_t)max_sites * 16 + 1024);
}

SparsePacker::~SparsePacker() {
    plane_free(reinterpret_cast<uint8_t*>(cells_), true); plane_free(reinterpret_cast<uint8_t*>(aux_), true);
    plane_free(reinterpret_cast<uint8_t*>(site_start_), true); plane_free(ref_, true);
}

void SparsePacker::grow(size_t want) {
    if (want <= cap_cells_) return;
    size_t cap = cap_cells_ ? cap_cells_ : 1024;
    while (cap < want) cap *= 2;
    uint32_t* c = reinterpret_cast<uint32_t*>(plane_alloc(cap * sizeof(uint32_t), true));
    uint32_t* a = reinterpret_cast<uint32_t*>(plane_alloc(cap * sizeof(uint32_t), true));
    if (n_cells_) { memcpy(c, cells_, n_cells_ * sizeof(uint32_t)); memcpy(a, aux_, n_cells_ * sizeof(uint32_t)); }
    plane_free(reinterpret_cast<uint8_t*>(cells_), true); plane_free(reinterpret_cast<uint8_t*>(aux_), true);
    cells_ = c; aux_ = a; cap_cells_ = cap;
}

void SparsePacker::begin_site(char ref_base) {
    if (n_sites_ >= max_sites_) throw std::runtime_error("[ERROR] SparsePacker is full");
    ref_[n_sites_] = (uint8_t)ref_base;
    ++n_sites_;
    site_start_[n_sites_] = (uint32_t)n_cells_;
}

void SparsePacker::add_cell(uint32_t sample, uint8_t base, uint8_t strand, uint8_t phred, uint8_t mapq, uint16_t rpr) {
    if (n_sites_ == 0) throw std::runtime_error("[ERROR] SparsePacker::add_cell before begin_site");
    if (sample >= n_samples_) throw std::runtime_error("[ERROR] SparsePacker: sample index out of range");
    if (n_cells_ >= 0xffffffffull) throw std::runtime_error("[ERROR] SparsePacker: more than 2^32 cells in one tile");
    grow(n_cells_ + 1);
    cells_[n_cells_] = BV_CELL_PACK(sample, base & 7u, strand & 3u, phred & 127u);
    aux_[n_cells_] = BV_CELL_AUX_PACK(mapq, rpr);
    ++n_cells_;
    site_start_[n_sites_] = (uint32_t)n_cells_;
}

bv_sparse_tile SparsePacker::tile() const {
    bv_sparse_tile t;
    t.cells = cells_; t.cells_aux = aux_; t.site_start = site_start_; t.ref_base = ref_; t.out = nullptr;
    t.n_sites = n_sites_; t.n_samples = n_samples_;
    t.format = BV_CELLS_U32; t.out_mode = BV_OUT_RECORDS;
    return t;
}

// ---- Context ----------------------------------------------------------------------------------------------------------
Context::Context(int device, float min_af, uint32_t max_samples, uint32_t max_sites, uint32_t n_slots, int em_abs_mode)
    : n_slots_(n_slots) {
    bv_params p;
    memset(&p, 0, sizeof(p));
    p.min_af = min_af;
    p.lrt_threshold = LRT_THRESHOLD;
    p.em_max_iter = 100;     // src/algorithm.h:213
    p.em_eps = 0.001f;       // src/algorithm.h:213
    p.em_abs_mode = em_abs_mode;
    p.max_samples = max_samples;
    p.max_sites = max_sites;
    p.n_slots = n_slots;
    check(bv_create(device, &p, &ctx_), nullptr, "bv_create");
    max_samples_ = max_samples;
    max_sites_ = max_sites;
    min_af_ = min_af;
    slot_tiles_.resize(n_slots);
}
Context::~Context() { bv_destroy(ctx_); }
void Context::submit(int slot, const bv_tile& tile) { check(bv_tile_submit(ctx_, slot, &tile), ctx_, "bv_tile_submit"); }
void Context::wait(int slot, bv_site_out* out) { check(bv_tile_wait(ctx_, slot, out), ctx_, "bv_tile_wait"); }
std::vector<bv_site_out> Context::run(const bv_tile& tile) {
    std::vector<bv_site_out> out(tile.n_sites);
    submit(0, tile);
    wait(0, out.data());
    return out;
}
void Context::submit(int slot, const bv_sparse_tile& tile) { check(bv_tile_submit_sparse(ctx_, slot, &tile), ctx_, "bv_tile_submit_sparse"); }
std::vector<bv_site_out> Context::run(const bv_sparse_tile& tile) {
    std::vector<bv_site_out> out(tile.n_sites);
    submit(0, tile);
    wait(0, out.data());
    return out;
}
void Context::submit_lists(int slot, const bv_tile& tile, const uint8_t (*lists)[4]) {
    check(bv_tile_submit_lists(ctx_, slot, &tile, lists), ctx_, "bv_tile_submit_lists");
    note_tile(slot, tile.n_sites, BV_OUT_RECORDS, tile.ref_base);
}
void Context::wait_lists(int slot, bv_site_out* out, bv_lrt_out* lrt_out) {
    check(bv_tile_wait_lists(ctx_, slot, out, lrt_out), ctx_, "bv_tile_wait_lists");
}
void Context::submit_lists(int slot, const bv_sparse_tile& tile, const uint8_t (*lists)[4]) {
    check(bv_tile_submit_sparse_lists(ctx_, slot, &tile, lists), ctx_, "bv_tile_submit_sparse_lists");
    note_tile(slot, tile.n_sites, (int)tile.out_mode, tile.ref_base);
}

void Context::note_tile(int slot, uint32_t n_sites, int out_mode, const uint8_t* ref_base) {
    SlotTile& st = slot_tiles_.at((size_t)slot);
    st.n_sites = n_sites; st.compact = out_mode == BV_OUT_COMPACT; st.ref_base = ref_base;
}

// the records part of a result: the compact views (and a copy of the REF bases they expand against), else nothing to do
void Context::take_records(int slot, TileResult& r, const bv_site_brief* brief, const bv_site_out* full, uint32_t n_full) {
    const SlotTile& st = slot_tiles_.at((size_t)slot);
    r.n_sites = st.n_sites;
    r.compact = st.compact;
    r.min_af = min_af_;
    if (!st.compact) return;
    r.brief = brief; r.full = full; r.n_full = n_full;
    if (st.n_sites) r.ref_base.assign(st.ref_base, st.ref_base + st.n_sites);
}

// the context's staging for what a wait copies out before TileResult gets its share: grown once, never zero-filled again
template <class T>
static T* staging(std::vector<T>& v, size_t n) {
    if (v.size() < n) v.resize(n);
    return v.data();
}

TileResult Context::wait_lists(int slot) {
    TileResult r;
    const SlotTile& st = slot_tiles_.at((size_t)slot);
    if (!st.compact) {
        r.records.resize(st.n_sites);
        r.lrt.resize(st.n_sites);
        check(bv_tile_wait_lists(ctx_, slot, r.records.data(), r.lrt.data()), ctx_, "bv_tile_wait_lists");
        take_records(slot, r, nullptr, nullptr, 0);
        return r;
    }
    const bv_site_brief* brief = nullptr;
    const bv_site_out* full = nullptr;
    uint32_t n_full = 0, n_lrt = 0;
    const bv_lrt_out* lrt = staging(lrt_stage_, st.n_sites);
    check(bv_tile_wait_lists_compact(ctx_, slot, &brief, &full, &n_full, lrt_stage_.data(), st.n_sites, &n_lrt), ctx_,
          "bv_tile_wait_lists_compact");
    r.lrt.assign(lrt, lrt + n_lrt);
    take_records(slot, r, brief, full, n_full);
    return r;
}

void Context::set_groups(const std::map<std::string, std::vector<size_t>>& group_smp_idx) {
    if (group_smp_idx.size() > BV_MAX_GROUPS)
        throw std::invalid_argument("[ERROR] set_groups: more than " + std::to_string(BV_MAX_GROUPS) + " population groups");
    std::vector<uint8_t> sg(max_samples_, (uint8_t)BV_GROUP_NONE);
    uint32_t g = 0;
    for (const auto& kv : group_smp_idx) {   // std::map: ascending name, the reference's order
        for (size_t i : kv.second) {
            if (i >= max_samples_)
                throw std::invalid_argument("[ERROR] set_groups: sample " + std::to_string(i) + " of group " + kv.first + " is out of range");
            if (sg[i] != BV_GROUP_NONE)
                throw std::invalid_argument("[ERROR] set_groups: sample " + std::to_string(i) + " is listed twice");
            sg[i] = (uint8_t)g;
        }
        ++g;
    }
    check(bv_set_groups(ctx_, sg.data(), max_samples_, g), ctx_, "bv_set_groups");
    n_groups_ = g;
}

void Context::submit_calls(int slot, const bv_tile& tile, const bv_tile_aux& aux) {
    check(bv_tile_submit_calls(ctx_, slot, &tile, &aux), ctx_, "bv_tile_submit_calls");
    note_tile(slot, tile.n_sites, tile.location == BV_LOC_HOST ? tile.out_mode : BV_OUT_RECORDS, tile.ref_base);
}

void Context::submit_calls(int slot, const bv_sparse_tile& tile) {
    check(bv_tile_submit_sparse_calls(ctx_, slot, &tile), ctx_, "bv_tile_submit_sparse_calls");
    note_tile(slot, tile.n_sites, (int)tile.out_mode, tile.ref_base);
}

TileResult Context::wait_calls(int slot) {
    TileResult r;
    const SlotTile& st = slot_tiles_.at((size_t)slot);
    const bv_call_out* calls = staging(calls_stage_, st.n_sites);
    const bv_group_out* groups = staging(groups_stage_, (size_t)st.n_sites * n_groups_);
    uint32_t n_calls = 0;
    bv_group_out* gp = n_groups_ ? groups_stage_.data() : nullptr;
    if (st.compact) {
        const bv_site_brief* brief = nullptr;
        const bv_site_out* full = nullptr;
        uint32_t n_full = 0;
        check(bv_tile_wait_calls_compact(ctx_, slot, &brief, &full, &n_full, calls_stage_.data(), st.n_sites, &n_calls, gp), ctx_,
              "bv_tile_wait_calls_compact");
        take_records(slot, r, brief, full, n_full);
    } else {
        r.records.resize(st.n_sites);
        check(bv_tile_wait_calls(ctx_, slot, r.records.data(), calls_stage_.data(), st.n_sites, &n_calls, gp), ctx_, "bv_tile_wait_calls");
        take_records(slot, r, nullptr, nullptr, 0);
    }
    // the device lists the called sites in no particular order: ascending site, groups alongside
    std::vector<uint32_t> order(n_calls);
    for (uint32_t k = 0; k < n_calls; ++k) order[k] = k;
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return calls[a].site < calls[b].site; });
    r.n_groups = n_groups_;
    r.calls.resize(n_calls);
    r.groups.resize((size_t)n_calls * n_groups_);
    for (uint32_t k = 0; k < n_calls; ++k) {
        r.calls[k] = calls[order[k]];
        for (uint32_t g = 0; g < n_groups_; ++g) r.groups[(size_t)k * n_groups_ + g] = groups[(size_t)order[k] * n_groups_ + g];
    }
    return r;
}

// ---- TileResult -------------------------------------------------------------------------------------------------------
bv_site_out TileResult::record(uint32_t site) const {
    if (site >= n_sites) throw std::out_of_range("[ERROR] TileResult::record: site out of range");
    if (!compact) return records[site];
    const bv_site_brief& b = brief[site];
    if (b.w0 & 0x80000000u) {
        const uint32_t k = b.w0 & 0x7fffffffu;
        if (k >= n_full) throw std::runtime_error("[ERROR] TileResult::record: compact record index out of range");
        return full[k];
    }
    bv_site_out rec;
    bv_site_expand(&b, ref_base[site], min_af, &rec);
    return rec;
}

const bv_call_out* TileResult::call(uint32_t site) const {
    auto it = std::lower_bound(calls.begin(), calls.end(), site, [](const bv_call_out& c, uint32_t s) { return c.site < s; });
    return it != calls.end() && it->site == site ? &*it : nullptr;
}

const bv_group_out* TileResult::group(uint32_t site, uint32_t g) const {
    const bv_call_out* c = call(site);
    if (!c || g >= n_groups) return nullptr;
    return &groups[(size_t)(c - calls.data()) * n_groups + g];
}

uint64_t Context::launch_count() const { return bv_launch_count(ctx_); }
double Context::fisher_fs(int ref_fwd, int ref_rev, int alt_fwd, int alt_rev) {
    const int32_t t[4] = {ref_fwd, ref_rev, alt_fwd, alt_rev};
    double fs = 0.0;
    check(bv_fisher_fs(ctx_, t, 1, &fs), ctx_, "bv_fisher_fs");
    return fs;
}

void Context::ranksum_test(const uint8_t* bases, const int32_t* values, const uint64_t* start, const uint8_t* ref_base,
                           const uint8_t* alt_mask, uint32_t n, double* phred_out) {
    check(bv_ranksum_test(ctx_, bases, values, start, ref_base, alt_mask, n, phred_out), ctx_, "bv_ranksum_test");
}

// ---- BaseType ---------------------------------------------------------------------------------------------------------
BaseType::BaseType(const BatchInfo* bi, const bv_site_out& rec)
    : ref_id_(bi->ref_id), ref_base_(bi->ref_base), ref_pos_(bi->ref_pos), rec_(rec) {
    fill_from_record();
    lrt_done_ = true;
}

BaseType::BaseType(const BatchInfo* bi, const bv_group_out& g) : ref_id_(bi->ref_id), ref_base_(bi->ref_base), ref_pos_(bi->ref_pos) {
    fill_alts(g.flags, g.n_alt, g.alt, g.af);
}

BaseType::BaseType(const BatchInfo* bi, const bv_lrt_out& lo) : ref_id_(bi->ref_id), ref_base_(bi->ref_base), ref_pos_(bi->ref_pos) {
    fill_alts(lo.flags, lo.n_alt, lo.alt, lo.af);
    var_qual_ = lo.qual;
}

// ALT set and AFs of an lrt(list) result (bv_lrt_out, bv_group_out)
void BaseType::fill_alts(uint8_t flags, int n_alt, const uint8_t* alt, const double* af) {
    if (flags & BV_FLAG_ZERO_SUBSET)   // src/basetype.cpp:113-115
        throw std::runtime_error("[ERROR] The sum of frequence of active bases must always > 0. Check: ");
    alt_bases_.clear();
    af_by_lrt_.clear();
    for (int k = 0; k < n_alt && k < 4; ++k) {
        const char b = BASES[alt[k] & 3];
        alt_bases_.push_back(b);
        af_by_lrt_[b] = af[k];
    }
    lrt_done_ = true;
}

namespace {
struct OneSite {   // the calling thread's default context for the one-site drop-in constructor
    std::unique_ptr<Context> ctx;
    std::unique_ptr<TilePacker> packer;
    float min_af = -1.f;
    uint32_t n = 0;
};
thread_local OneSite t_one;

// the calling thread's one-site context and packer, made fit for min_af `maf` and rows of n samples
void one_site_prepare(float maf, uint32_t n) {
    if (!t_one.ctx || t_one.min_af != maf || t_one.n < n) {
        const char* d = getenv("BASEVAR_B200_DEVICE");
        t_one.ctx.reset();
        t_one.packer.reset();
        const uint32_t cap = std::max<uint32_t>(n, 1);
        t_one.ctx.reset(new Context(d ? atoi(d) : 0, maf, cap, 1, 1));
        t_one.min_af = maf;
        t_one.n = cap;
    }
    if (!t_one.packer || t_one.packer->n_samples() != n) t_one.packer.reset(new TilePacker(n, 1));
    t_one.packer->clear();
}
}  // namespace

BaseType::BaseType(const BatchInfo* bi, double af)
    : ref_id_(bi->ref_id), ref_base_(bi->ref_base), ref_pos_(bi->ref_pos) {
    const float maf = (float)af;
    const uint32_t n = (uint32_t)bi->n;
    one_site_prepare(maf, n);
    t_one.packer->add_site(*bi);   // throws on a malformed base string, like the reference's constructor
    const bv_tile t = t_one.packer->tile();
    rec_ = t_one.ctx->run(t)[0];
    row_base_.assign(t.base, t.base + n);
    row_qual_.assign(t.qual, t.qual + n);
    row_strand_.assign(t.strand, t.strand + n);
    row_ref_ = (char)t.ref_base[0];
    min_af_ = maf;
    has_row_ = true;
    // the constructor gives depths; ALT / AF / QUAL appear with lrt() (src/basetype.cpp:130)
    total_depth_ = (int)(rec_.depth[0] + rec_.depth[1] + rec_.depth[2] + rec_.depth[3] + rec_.depth_other);
}

void BaseType::lrt(const std::vector<char>& specific_bases) {
    if (specific_bases != BASES) {
        if (!has_row_)
            throw std::invalid_argument("[ERROR] lrt() over a list other than A,C,G,T needs the site's reads: build the BaseType "
                                        "from a BatchInfo and min_af");
        lrt_list(specific_bases);
        return;
    }
    if (rec_.flags & BV_FLAG_ZERO_SUBSET)   // src/basetype.cpp:113-115
        throw std::runtime_error("[ERROR] The sum of frequence of active bases must always > 0. Check: ");
    if (lrt_done_) return;   // (the reference appends the ALT alleles again on a second call; nobody relies on that)
    fill_from_record();
    lrt_done_ = true;
}

void BaseType::lrt_list(const std::vector<char>& specific_bases) {
    uint8_t list[1][4] = {{BV_LIST_END, BV_LIST_END, BV_LIST_END, BV_LIST_END}};
    int n = 0;
    for (size_t i = 0; i < specific_bases.size(); ++i) {
        const char c = specific_bases[i];
        for (size_t j = 0; j < i; ++j)
            if (specific_bases[j] == c) throw std::invalid_argument(std::string("[ERROR] lrt(): base '") + c + "' is listed twice");
        const int code = c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1;
        if (code >= 0) list[0][n++] = (uint8_t)code;   // any other character has no depth entry: never active (basetype.cpp:137)
    }
    const uint32_t N = (uint32_t)row_base_.size();
    one_site_prepare(min_af_, N);
    t_one.packer->add_site_cells(row_ref_, row_base_.data(), row_qual_.data(), row_strand_.data(), nullptr);
    bv_lrt_out lo;
    t_one.ctx->submit_lists(0, t_one.packer->tile(), list);
    t_one.ctx->wait_lists(0, nullptr, &lo);
    fill_alts(lo.flags, lo.n_alt, lo.alt, lo.af);
    var_qual_ = lo.qual;
}

void BaseType::fill_from_record() {
    total_depth_ = (int)(rec_.depth[0] + rec_.depth[1] + rec_.depth[2] + rec_.depth[3] + rec_.depth_other);
    alt_bases_.clear();
    af_by_lrt_.clear();
    for (int k = 0; k < rec_.n_alt && k < 4; ++k) {
        const char b = BASES[rec_.alt[k] & 3];
        alt_bases_.push_back(b);
        af_by_lrt_[b] = rec_.af[k];
    }
    var_qual_ = rec_.qual;
}

double BaseType::get_base_depth(char b) const {
    for (size_t i = 0; i < BASES.size(); ++i)
        if (BASES[i] == b) return (double)rec_.depth[i];
    throw std::runtime_error(std::string("[ERROR] out_of_range:: map::at '") + b + "' not found.");
}

double BaseType::get_lrt_af(char b) const {
    std::map<char, double>::const_iterator it = af_by_lrt_.find(b);
    if (it == af_by_lrt_.end()) throw std::runtime_error(std::string("[ERROR] out_of_range:: map::at '") + b + "' not found.");
    return it->second;
}

// The calling thread's default context for the free functions, made again when it has room for fewer than max_samples samples.
static Context* thread_context(uint32_t max_samples) {
    if (!t_one.ctx || t_one.ctx->max_samples() < max_samples) {
        const char* d = getenv("BASEVAR_B200_DEVICE");
        t_one.ctx.reset();
        t_one.packer.reset();
        t_one.n = std::max<uint32_t>(max_samples, 1);
        t_one.min_af = 0.01f;
        t_one.ctx.reset(new Context(d ? atoi(d) : 0, t_one.min_af, t_one.n, 1, 1));
    }
    return t_one.ctx.get();
}

// ---- strand_bias -------------------------------------------------------------------------------------------------------
static int code_of(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }

StrandBiasInfo strand_bias(const char ref_base, const std::string alt_bases_string, const bv_site_out& rec, Context* ctx) {
    if (rec.flags & BV_FLAG_BAD_STRAND)   // src/basetype.cpp:271-273
        throw std::runtime_error("[ERROR] Get strange strand symbol: ");
    StrandBiasInfo s;
    const int rc = code_of(ref_base);
    s.ref_fwd = rc >= 0 ? (int)rec.fwd[rc] : 0;
    s.ref_rev = rc >= 0 ? (int)rec.rev[rc] : 0;
    s.alt_fwd = s.alt_rev = 0;
    unsigned alt_set = 0;
    for (char c : alt_bases_string) {
        const int k = code_of(c);
        if (k < 0 || k == rc || (alt_set >> k & 1)) continue;   // a base equal to REF counts as REF (basetype.cpp:256-261)
        alt_set |= 1u << k;
        s.alt_fwd += (int)rec.fwd[k];
        s.alt_rev += (int)rec.rev[k];
    }
    unsigned cvg_set = 0xfu & ~(rc >= 0 ? 1u << rc : 0u), vcf_set = 0;
    for (int k = 0; k < rec.n_alt && k < 4; ++k) vcf_set |= 1u << (rec.alt[k] & 3);
    // bases without reads do not change the table
    unsigned covered = 0;
    for (int k = 0; k < 4; ++k) if (rec.fwd[k] + rec.rev[k]) covered |= 1u << k;
    if (((alt_set ^ cvg_set) & covered) == 0) s.fs = rec.fs_cvg;
    else if (rec.n_alt && ((alt_set ^ vcf_set) & covered) == 0) s.fs = rec.fs_vcf;
    else if ((s.alt_fwd | s.alt_rev) == 0 || (s.ref_fwd | s.ref_rev) == 0) s.fs = 0.0;   // one possible table: p == 1
    else {
        // neither of the two sets the record carries FS for: the 2x2 table goes to the device (bv_fisher_fs, the code of bv_fisher_kernel)
        const uint32_t reads = (uint32_t)(s.ref_fwd + s.ref_rev + s.alt_fwd + s.alt_rev);
        if (!ctx) ctx = thread_context(reads - 1);   // the log-factorial table covers max_samples + 1 reads
        s.fs = ctx->fisher_fs(s.ref_fwd, s.ref_rev, s.alt_fwd, s.alt_rev);
    }
    // src/basetype.cpp:286, int32 products as in the reference
    s.sor = (s.ref_rev * s.alt_fwd > 0) ? (double)(s.ref_fwd * s.alt_rev) / (double)(s.ref_rev * s.alt_fwd) : 10000;
    return s;
}

// ---- ref_vs_alt_ranksumtest ---------------------------------------------------------------------------------------------
static double ranksum_one(const char ref_base, const std::string& alt_bases_string, const std::vector<char>& bases,
                          const std::vector<int32_t>& values, Context* ctx) {
    if (ref_base >= 'a' && ref_base <= 'z')
        throw std::invalid_argument(std::string("[ERROR] ref_vs_alt_ranksumtest: lowercase ref_base '") + ref_base + "'");
    uint8_t alt_mask = 0;
    for (char c : alt_bases_string) {
        const int k = code_of(c);
        if (k < 0) throw std::invalid_argument(std::string("[ERROR] ref_vs_alt_ranksumtest: ALT base '") + c + "' is not A/C/G/T");
        alt_mask |= (uint8_t)(1u << k);
    }
    const bool ref_is_code = code_of(ref_base) >= 0 || ref_base == 'N';
    std::vector<uint8_t> codes(bases.size());
    for (size_t i = 0; i < bases.size(); ++i) {
        const char c = bases[i];
        if (!ref_is_code && c == ref_base)
            throw std::invalid_argument(std::string("[ERROR] ref_vs_alt_ranksumtest: ref_base '") + ref_base +
                                        "' is not A/C/G/T/N and a base equals it");
        const int k = code_of(c);
        codes[i] = (uint8_t)(k >= 0 ? k : c == 'N' ? BV_BASE_N : c == '+' ? BV_BASE_INS : c == '-' ? BV_BASE_DEL : BV_BASE_OTHER);
    }
    const uint32_t n = (uint32_t)bases.size();
    if (!ctx) ctx = thread_context(n);
    const uint64_t start[2] = {0, n};
    const uint8_t ref = (uint8_t)ref_base;
    double v = 0.0;
    ctx->ranksum_test(codes.data(), values.data(), start, &ref, &alt_mask, 1, &v);
    return v;
}

double ref_vs_alt_ranksumtest(const char ref_base, const std::string alt_bases_string, const std::vector<char>& bases,
                              const std::vector<int>& values, Context* ctx) {
    if (bases.size() != values.size()) throw std::invalid_argument("[ERROR] ref_vs_alt_ranksumtest: bases and values differ in size");
    return ranksum_one(ref_base, alt_bases_string, bases, std::vector<int32_t>(values.begin(), values.end()), ctx);
}

double ref_vs_alt_ranksumtest(const char ref_base, const std::string alt_bases_string, const std::vector<char>& bases,
                              const std::vector<char>& values, Context* ctx) {
    if (bases.size() != values.size()) throw std::invalid_argument("[ERROR] ref_vs_alt_ranksumtest: bases and values differ in size");
    std::vector<int32_t> v(values.size());
    for (size_t i = 0; i < values.size(); ++i) v[i] = (int32_t)(signed char)values[i];   // as g++ on x86-64 widens a char
    return ranksum_one(ref_base, alt_bases_string, bases, v, ctx);
}

// ---- region sharding ----------------------------------------------------------------------------------------------------
std::vector<Shard> shard_region(uint64_t reg_beg, uint64_t reg_end, int n_gpus, uint64_t step) {
    std::vector<Shard> out;
    if (reg_end <= reg_beg || n_gpus <= 0) return out;
    if (step == 0) step = 1;
    const uint64_t n_steps = (reg_end - reg_beg + step - 1) / step;   // 100-kb tasks, the last one may be short
    const uint64_t g = std::min<uint64_t>((uint64_t)n_gpus, n_steps);
    uint64_t s0 = 0;
    for (uint64_t i = 0; i < g; ++i) {
        const uint64_t cnt = n_steps / g + (i < n_steps % g ? 1 : 0);
        Shard sh;
        sh.gpu = (int)i;
        sh.beg = reg_beg + s0 * step;
        sh.end = std::min(reg_end, reg_beg + (s0 + cnt) * step);
        out.push_back(sh);
        s0 += cnt;
    }
    return out;
}

void run_region(uint64_t reg_beg, uint64_t reg_end, const RunOptions& opt, const TileSource& fill, const RecordSink& sink) {
    std::vector<int> devices = opt.devices;
    if (devices.empty()) {
        // probe: contexts on devices 0,1,... until creation fails
        for (int d = 0; d < 64; ++d) {
            bv_params p;
            memset(&p, 0, sizeof(p));
            p.min_af = opt.min_af; p.lrt_threshold = LRT_THRESHOLD; p.em_max_iter = 100; p.em_eps = 0.001f; p.max_samples = 1;
            bv_ctx* c = nullptr;
            if (bv_create(d, &p, &c) != BV_OK) break;
            bv_destroy(c);
            devices.push_back(d);
        }
        if (devices.empty()) throw std::runtime_error(std::string("[ERROR] no CUDA device: ") + bv_last_error(nullptr));
    }
    const int n_shards = opt.n_shards > 0 ? opt.n_shards : (int)devices.size();
    const std::vector<Shard> shards = shard_region(reg_beg, reg_end, n_shards);
    std::vector<std::vector<bv_site_out>> results(shards.size());
    std::vector<std::exception_ptr> errors(shards.size());
    std::vector<std::thread> workers;
    for (size_t si = 0; si < shards.size(); ++si) {
        workers.emplace_back([&, si]() {
            try {
                const Shard& sh = shards[si];
                const uint32_t n_slots = std::max<uint32_t>(opt.n_slots, 1);
                Context ctx(devices[si % devices.size()], opt.min_af, opt.n_samples, opt.tile_sites, n_slots, opt.em_abs_mode);
                std::vector<std::unique_ptr<TilePacker>> packers;
                for (uint32_t k = 0; k < n_slots; ++k) packers.emplace_back(new TilePacker(opt.n_samples, opt.tile_sites));
                std::vector<bv_site_out>& res = results[si];
                res.resize(sh.end - sh.beg);
                struct Pending { uint64_t site0; uint32_t n; };
                std::vector<Pending> pending(n_slots, Pending{0, 0});
                uint32_t slot = 0;
                for (uint64_t s0 = sh.beg; s0 < sh.end; s0 += opt.tile_sites) {
                    const uint32_t n = (uint32_t)std::min<uint64_t>(opt.tile_sites, sh.end - s0);
                    if (pending[slot].n) {   // the slot's previous tile: collect before its packer is reused
                        ctx.wait((int)slot, res.data() + (pending[slot].site0 - sh.beg));
                        pending[slot].n = 0;
                    }
                    TilePacker& pk = *packers[slot];
                    pk.clear();
                    fill(s0, n, pk);
                    if (pk.n_sites() != n) throw std::runtime_error("[ERROR] TileSource packed a wrong number of sites");
                    ctx.submit((int)slot, pk.tile());
                    pending[slot] = Pending{s0, n};
                    slot = (slot + 1) % n_slots;
                }
                for (uint32_t k = 0; k < n_slots; ++k) {
                    const uint32_t sl = (slot + k) % n_slots;
                    if (pending[sl].n) ctx.wait((int)sl, res.data() + (pending[sl].site0 - sh.beg));
                }
            } catch (...) {
                errors[si] = std::current_exception();
            }
        });
    }
    for (auto& w : workers) w.join();
    for (auto& e : errors)
        if (e) std::rethrow_exception(e);   // like future.get() in the reference (basetype_caller.cpp:513-517)
    // merge = concatenation in coordinate order (the reference's merge_file_by_line order, basetype_utils.cpp:90-123)
    for (size_t si = 0; si < shards.size(); ++si)
        for (uint64_t s0 = shards[si].beg; s0 < shards[si].end; s0 += opt.tile_sites) {
            const uint32_t n = (uint32_t)std::min<uint64_t>(opt.tile_sites, shards[si].end - s0);
            sink(s0, results[si].data() + (s0 - shards[si].beg), n);
        }
}

}  // namespace bvhost
