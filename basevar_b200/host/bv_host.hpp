// bv_host.hpp -- C++ host layer over the C ABI (include/basevar_b200.h): the reference-facing side of the drop-in.
//
// It mirrors the interface the reference's per-site driver uses (same names, argument meaning and error behaviour):
//
//   reference (src/basetype.h)                              here (namespace bvhost)
//   -----------------------------------------------------   ---------------------------------------------------------
//   struct BatchInfo                      :25-43            BatchInfo (same members)
//   struct StrandBiasInfo                 :56-61            StrandBiasInfo (same members)
//   class BaseType, ctor + lrt() + getters :64-153          BaseType: filled from a device record (batch path), or
//                                                           BaseType(const BatchInfo*, double) + lrt() for one site
//   strand_bias(ref, alts, bases, strands) :178-181         strand_bias(ref, alts, record)
//   ref_vs_alt_ranksumtest(...)           :168-176          ref_vs_alt_ranksumtest (same arguments; bv_ranksum_test)
//   BatchInfo rows -> BaseType per site,                    TilePacker (BatchInfo -> packed SoA planes in pinned memory)
//     src/basetype_caller.cpp:686-743                       Context (slots: H2D copy, kernels, D2H copy per tile)
//   100-kb tasks over a ThreadPool,                         shard_region / run_region: contiguous region shards, one host
//     src/basetype_caller.cpp:469-525                       worker + context per GPU, records delivered in coordinate order
//
// All the arithmetic happens on the GPU behind the C ABI; nothing here computes likelihoods, EM, LRT or Fisher.
#pragma once
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/basevar_b200.h"

namespace bvhost {

static const std::vector<char> BASES = {'A', 'C', 'G', 'T'};   // src/basetype.h:19
static const int LRT_THRESHOLD = 24;                           // src/basetype.h:21
static const int QUAL_THRESHOLD = 20;                          // src/basetype.h:22

struct BatchInfo {   // src/basetype.h:25-43
    size_t n;
    std::string ref_id;
    std::string ref_base;
    uint32_t ref_pos;
    uint32_t depth;
    std::vector<std::string> align_bases;
    std::vector<char> align_base_quals;
    std::vector<int> mapqs;
    std::vector<char> map_strands;
    std::vector<int> base_pos_ranks;
    BatchInfo() : n(0), ref_pos(0), depth(0) {}
};

struct StrandBiasInfo {   // src/basetype.h:56-61
    int ref_fwd, ref_rev;
    int alt_fwd, alt_rev;
    double fs;
    double sor;
};

// ---- cell encoding ---------------------------------------------------------------------------------------------------
// First character of align_bases[i] -> BV_BASE_* (src/basetype.cpp:50-56).  A multi-character string that is not an
// indel makes the reference throw; so does this.
uint8_t encode_base(const std::string& align_base);
inline uint8_t encode_strand(char c) { return c == '+' ? BV_STRAND_FWD : c == '-' ? BV_STRAND_REV : BV_STRAND_NONE; }
// min(100.0f / n_bam, min_af) in float (src/basetype_caller.cpp:122)
float cli_min_af(float min_af, size_t n_bam);

// ---- pinned planes + packer ------------------------------------------------------------------------------------------
class TilePacker {
public:
    TilePacker(uint32_t n_samples, uint32_t max_sites, bool pinned = true);
    ~TilePacker();
    TilePacker(const TilePacker&) = delete;
    TilePacker& operator=(const TilePacker&) = delete;

    void clear() { n_sites_ = 0; }
    uint32_t n_sites() const { return n_sites_; }
    uint32_t n_samples() const { return n_samples_; }
    uint32_t capacity() const { return max_sites_; }
    uint64_t pitch() const { return pitch_; }

    // One site from the reference's per-site struct (any type with BatchInfo's members).
    template <class BI>
    void add_site(const BI& bi) {
        if (bi.n != n_samples_) throw std::runtime_error("[ERROR] BatchInfo::n does not match the tile's sample count");
        uint8_t *b, *q, *s, *m;
        next_row(bi.ref_base.empty() ? 'N' : bi.ref_base[0], &b, &q, &s, &m);
        uint16_t* r = rpr_ + (size_t)(n_sites_ - 1) * pitch_;
        for (size_t i = 0; i < bi.n; ++i) {
            b[i] = encode_base(bi.align_bases[i]);
            q[i] = (uint8_t)(bi.align_base_quals[i] - 33);
            s[i] = encode_strand(bi.map_strands[i]);
            m[i] = (uint8_t)(bi.mapqs[i] > 255 ? 255 : bi.mapqs[i] < 0 ? 0 : bi.mapqs[i]);
            const int rp = bi.base_pos_ranks.empty() ? 0 : bi.base_pos_ranks[i];   // clamped as SparsePacker::add_site does
            r[i] = (uint16_t)(rp < 0 ? 0 : rp > 65535 ? 65535 : rp);
        }
    }
    // One site of already encoded cells (row pointers of n_samples bytes each; mapq may be null).
    void add_site_cells(char ref_base, const uint8_t* base, const uint8_t* qual, const uint8_t* strand, const uint8_t* mapq);
    // Raw row access for packers that scatter per-sample runs (rows are pre-filled with uncovered cells).
    void next_row(char ref_base, uint8_t** base, uint8_t** qual, uint8_t** strand, uint8_t** mapq);

    bv_tile tile() const;   // BV_LOC_HOST tile over the packed sites
    // the called-site kernels' planes of the same sites: mapqs, and base_pos_ranks clamped to 0..65535 (rows next_row() /
    // add_site_cells() start are all zero); rpr_pitch = pitch()
    bv_tile_aux aux() const;
    const uint8_t* mapq_plane() const { return mapq_; }

private:
    uint32_t n_samples_, max_sites_, n_sites_ = 0;
    uint64_t pitch_;
    bool pinned_;
    uint8_t *base_ = nullptr, *qual_ = nullptr, *strand_ = nullptr, *mapq_ = nullptr, *ref_ = nullptr;
    uint16_t* rpr_ = nullptr;
};

// ---- sparse packer: only the covered cells of a site travel (bv_sparse_tile) ----------------------------------------------
// What a pileup produces at < 1x depth: one packed word per (sample, position) a read covers.  A sample whose entry is
// the reference's filler for "no read here" (`N`, `!`, strand `.`; src/basetype_caller.cpp:1063-1075) adds nothing.
class SparsePacker {
public:
    SparsePacker(uint32_t n_samples, uint32_t max_sites, size_t reserve_cells = 0);
    ~SparsePacker();
    SparsePacker(const SparsePacker&) = delete;
    SparsePacker& operator=(const SparsePacker&) = delete;

    void clear() { n_sites_ = 0; n_cells_ = 0; }
    uint32_t n_sites() const { return n_sites_; }
    size_t n_cells() const { return n_cells_; }

    void begin_site(char ref_base);                                      // then add_cell() for its covered samples
    void add_cell(uint32_t sample, uint8_t base, uint8_t strand, uint8_t phred, uint8_t mapq = 0, uint16_t rpr = 0);
    template <class BI>
    void add_site(const BI& bi) {   // the reference's per-site struct (any type with BatchInfo's members)
        if (bi.n != n_samples_) throw std::runtime_error("[ERROR] BatchInfo::n does not match the tile's sample count");
        begin_site(bi.ref_base.empty() ? 'N' : bi.ref_base[0]);
        for (size_t i = 0; i < bi.n; ++i) {
            const uint8_t b = encode_base(bi.align_bases[i]), st = encode_strand(bi.map_strands[i]);
            const uint8_t q = (uint8_t)(bi.align_base_quals[i] - 33);
            const int mq = bi.mapqs[i] > 255 ? 255 : bi.mapqs[i] < 0 ? 0 : bi.mapqs[i];
            const int rp = bi.base_pos_ranks.empty() ? 0 : bi.base_pos_ranks[i];
            if (b == BV_BASE_N && q == 0 && st == BV_STRAND_NONE && mq == 0 && rp == 0) continue;
            add_cell((uint32_t)i, b, st, q, (uint8_t)mq, (uint16_t)(rp < 0 ? 0 : rp > 65535 ? 65535 : rp));
        }
    }
    bv_sparse_tile tile() const;   // valid until the next clear() / add

private:
    void grow(size_t want);
    uint32_t n_samples_, max_sites_, n_sites_ = 0;
    size_t n_cells_ = 0, cap_cells_ = 0;
    uint32_t *cells_ = nullptr, *aux_ = nullptr, *site_start_ = nullptr;   // pinned
    uint8_t* ref_ = nullptr;
};

// ---- the batch results of one tile --------------------------------------------------------------------------------------
// What Context::wait_calls / wait_lists collect: the records (all of them, or the compact form), the called-site outputs and
// the list results.  The compact views point into the slot's pinned staging: valid until the slot's next submit.
struct TileResult {
    uint32_t n_sites = 0;
    bool compact = false;
    std::vector<bv_site_out> records;        // BV_OUT_RECORDS: one per site
    const bv_site_brief* brief = nullptr;    // BV_OUT_COMPACT: one per site (bv_tile_wait_compact) ...
    const bv_site_out* full = nullptr;       // ... and the n_full records they point into
    uint32_t n_full = 0;
    std::vector<uint8_t> ref_base;           // BV_OUT_COMPACT: the tile's REF bases, for bv_site_expand
    float min_af = 0.f;
    std::vector<bv_call_out> calls;          // called sites (n_alt > 0), ascending site
    uint32_t n_groups = 0;
    std::vector<bv_group_out> groups;        // [calls.size()][n_groups], groups[k * n_groups + g] belongs to calls[k]
    std::vector<bv_lrt_out> lrt;             // lists tiles: one per site (BV_OUT_RECORDS), or one per site whose list is
                                             // non-empty, in site order (BV_OUT_COMPACT)

    bv_site_out record(uint32_t site) const;                      // the site's record (all-REF sites expanded)
    const bv_call_out* call(uint32_t site) const;                 // null when the site is not called
    const bv_group_out* group(uint32_t site, uint32_t g) const;   // null when the site is not called
};

// ---- results of a device-resident tile ---------------------------------------------------------------------------------
// The device buffers of one tile whose pileup is already in GPU memory (Context::run_device): the fields of bv_device_out
// (include/basevar_b200.h), all null but kind / out_mode until set.  The caller owns the buffers (cudaMalloc or any device
// allocator); the mirror never touches device memory itself.
struct DeviceResult : bv_device_out {
    explicit DeviceResult(int kind_ = BV_RUN_PLAIN, int out_mode_ = BV_OUT_RECORDS) : bv_device_out() {
        kind = kind_;
        out_mode = out_mode_;
    }
};

// ---- a context bound to one GPU ---------------------------------------------------------------------------------------
class Context {
public:
    Context(int device, float min_af, uint32_t max_samples, uint32_t max_sites, uint32_t n_slots = 2,
            int em_abs_mode = BV_EM_ABS_INT_TRUNC);
    ~Context();
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;

    void submit(int slot, const bv_tile& tile);          // asynchronous; throws std::runtime_error on failure
    void wait(int slot, bv_site_out* out);               // blocks; `out` receives the tile's records
    std::vector<bv_site_out> run(const bv_tile& tile);   // submit + wait on slot 0
    void submit(int slot, const bv_sparse_tile& tile);   // sparse transport of the same tile (kernel K0 expands it)
    std::vector<bv_site_out> run(const bv_sparse_tile& tile);
    // the same plus BaseType::lrt(list) per site (bv_tile_submit_lists): lists[n_sites][4], BV_LIST_END-terminated
    void submit_lists(int slot, const bv_tile& tile, const uint8_t (*lists)[4]);
    void wait_lists(int slot, bv_site_out* out, bv_lrt_out* lrt_out);
    // sparse tiles (bv_tile_submit_sparse_lists), BV_OUT_RECORDS or BV_OUT_COMPACT (tile.out_mode); cells_aux is not read
    void submit_lists(int slot, const bv_sparse_tile& tile, const uint8_t (*lists)[4]);
    TileResult wait_lists(int slot);   // records or compact view, and `lrt`
    // Population groups of the called-site kernels (bv_set_groups), as _out_vcf_line's group_smp_idx holds them: group g is the
    // g-th name in map order (ascending, as basetype_caller.cpp:756 iterates them); samples in no group belong to none.
    // std::invalid_argument: more than BV_MAX_GROUPS groups, a sample listed twice, a sample index >= max_samples.
    void set_groups(const std::map<std::string, std::vector<size_t>>& group_smp_idx);
    uint32_t n_groups() const { return n_groups_; }
    // The VCF row's batch outputs (bv_tile_submit_calls / bv_tile_submit_sparse_calls): rank sums and population groups of
    // every called site.  BV_OUT_COMPACT (tile.out_mode) for host tiles; collect with wait_calls.
    void submit_calls(int slot, const bv_tile& tile, const bv_tile_aux& aux);
    void submit_calls(int slot, const bv_sparse_tile& tile);
    TileResult wait_calls(int slot);   // records or compact view, `calls` and `groups`
    // A pileup already in GPU memory: sparse cells (bv_tile_run_device_sparse) or dense planes (bv_tile_run_device_ex, with the
    // mapq / rpr planes in `aux` for BV_RUN_CALLS), every result into the device buffers `out` names.  `stream` is a
    // cudaStream_t; stream ordered, returns at once.  Throws std::runtime_error when the call is refused (nothing is queued then).
    void run_device(const bv_sparse_tile& tile, const DeviceResult& out, void* stream = nullptr);
    void run_device(const bv_tile& tile, const DeviceResult& out, void* stream = nullptr, const bv_tile_aux* aux = nullptr);
    uint32_t n_slots() const { return n_slots_; }
    uint64_t launch_count() const;
    bv_ctx* raw() { return ctx_; }
    uint32_t max_samples() const { return max_samples_; }
    // FS of free-standing 2x2 strand tables {ref_fwd, ref_rev, alt_fwd, alt_rev} on the device (bv_fisher_fs)
    double fisher_fs(int ref_fwd, int ref_rev, int alt_fwd, int alt_rev);
    // ref_vs_alt_ranksumtest of n free-standing problems on the device (bv_ranksum_test; arguments as there, host memory)
    void ranksum_test(const uint8_t* bases, const int32_t* values, const uint64_t* start, const uint8_t* ref_base,
                      const uint8_t* alt_mask, uint32_t n, double* phred_out);

private:
    struct SlotTile { uint32_t n_sites = 0; bool compact = false; const uint8_t* ref_base = nullptr; };
    void note_tile(int slot, uint32_t n_sites, int out_mode, const uint8_t* ref_base);
    void take_records(int slot, TileResult& r, const bv_site_brief* brief, const bv_site_out* full, uint32_t n_full);
    bv_ctx* ctx_ = nullptr;
    uint32_t n_slots_;
    uint32_t max_samples_ = 0;
    uint32_t max_sites_ = 0;
    float min_af_ = 0.f;
    uint32_t n_groups_ = 0;
    std::vector<SlotTile> slot_tiles_;
    // what the waits copy out of the slots before a TileResult takes the tile's share (sized by the largest tile waited for)
    std::vector<bv_call_out> calls_stage_;
    std::vector<bv_group_out> groups_stage_;
    std::vector<bv_lrt_out> lrt_stage_;
};

// ---- per-site mirror of the reference's class --------------------------------------------------------------------------
class BaseType {
public:
    BaseType() {}
    // Batch path: the record the device produced for this site.
    BaseType(const BatchInfo* smp_bi, const bv_site_out& rec);
    // Batch path of lrt(list): a population group's result (K6, TileResult::group) or a list's (K8, TileResult::lrt).  The
    // getters give the ALT set, get_lrt_af and (lists only; 0 for a group) get_var_qual as BaseType(&bi, af).lrt(list) does;
    // depths are not carried (get_total_depth 0).  Throws like lrt(list) when the EM met a zero-frequency subset.
    BaseType(const BatchInfo* smp_bi, const bv_group_out& group);
    BaseType(const BatchInfo* smp_bi, const bv_lrt_out& lrt);
    // Drop-in path (src/basetype.h:105): one site through a one-row tile on the calling thread's default context
    // (device BASEVAR_B200_DEVICE or 0).  `af` is the CLI's float min_af widened to double (basetype_caller.cpp:506).
    BaseType(const BatchInfo* smp_bi, double af);

    void lrt() { lrt(BASES); }                              // src/basetype.h:117
    // Any ordered list (src/basetype.h:118, the population-group path's lrt([REF, ALT...])): the site's row runs again with
    // the list on the calling thread's context (bv_tile_submit_lists).  A/C/G/T map to base codes; any other character is
    // never active (it has no depth entry).  A repeated character throws std::invalid_argument.  Needs the reads: a
    // BaseType built from a record alone throws std::invalid_argument for any list other than {A,C,G,T}.
    void lrt(const std::vector<char>& specific_bases);

    bool is_only_snp() const { return true; }
    const std::string& get_ref_id() const { return ref_id_; }
    const uint32_t& get_ref_pos() const { return ref_pos_; }
    const std::string& get_ref_base() const { return ref_base_; }
    const std::vector<char>& get_alt_bases() const { return alt_bases_; }
    double get_var_qual() const { return var_qual_; }
    int get_total_depth() const { return total_depth_; }
    double get_base_depth(char b) const;   // throws std::runtime_error for a key that is not A/C/G/T (basetype.h:127-139)
    double get_lrt_af(char b) const;       // throws std::runtime_error for a base that is not an ALT (basetype.h:141-151)
    const bv_site_out& record() const { return rec_; }

private:
    void fill_from_record();
    void fill_alts(uint8_t flags, int n_alt, const uint8_t* alt, const double* af);
    void lrt_list(const std::vector<char>& specific_bases);
    std::string ref_id_, ref_base_;
    uint32_t ref_pos_ = 0;
    std::vector<char> alt_bases_;
    std::map<char, double> af_by_lrt_;
    double var_qual_ = 0.0;
    int total_depth_ = 0;
    bool lrt_done_ = false;
    bv_site_out rec_{};
    // drop-in path: the site's encoded row, kept for lrt(list) (the reference's BatchInfo is only borrowed by the ctor)
    std::vector<uint8_t> row_base_, row_qual_, row_strand_;
    char row_ref_ = 'N';
    float min_af_ = 0.f;
    bool has_row_ = false;
};

// strand_bias(ref, ALT string) from a device record (src/basetype.cpp:244-295).  The counts come from the record's 2x4
// strand table for any ALT set; FS is read from the record for the two sets the reference asks for -- all non-REF bases (CVG
// row, basetype_caller.cpp:1236-1245) and the called ALT alleles (VCF row, :1164) -- and computed on the device for any other
// set (bv_fisher_fs; `ctx`, or the calling thread's default context, created on first use on device BASEVAR_B200_DEVICE or 0).
// A record flagged BV_FLAG_BAD_STRAND throws the reference's "[ERROR] Get strange strand symbol" error.
StrandBiasInfo strand_bias(const char ref_base, const std::string alt_bases_string, const bv_site_out& rec, Context* ctx = nullptr);

// ref_vs_alt_ranksumtest (src/basetype.h:168-176, src/basetype.cpp:201-242): -10 log10 of the two-sided Wilcoxon rank-sum p of
// the values of REF reads vs those of ALT reads, classified by the first character of each read's base, as a double (the
// caller truncates); 10000 when a class is empty or p == 0.  Computed on the device (bv_ranksum_test) on `ctx`, or on the
// calling thread's default context (device BASEVAR_B200_DEVICE or 0, made on first use and again for a longer list).
// Characters map to base codes: A/C/G/T, 'N', '+' (insertion), '-' (deletion), anything else BV_BASE_OTHER; N, indels and
// other characters are in neither class, a base equal to ref_base is a REF read, one in alt_bases_string an ALT read.
// The char overload widens each value as a signed char.  std::invalid_argument when bases and values differ in size.
// Departures from the reference, which compares raw characters where the packed codes cannot (std::invalid_argument):
//   - alt_bases_string holds a character other than A/C/G/T;
//   - ref_base is lowercase;
//   - ref_base is a character other than A/C/G/T/N and some entry of bases equals it.
double ref_vs_alt_ranksumtest(const char ref_base, const std::string alt_bases_string, const std::vector<char>& bases,
                              const std::vector<int>& values, Context* ctx = nullptr);
double ref_vs_alt_ranksumtest(const char ref_base, const std::string alt_bases_string, const std::vector<char>& bases,
                              const std::vector<char>& values, Context* ctx = nullptr);

// ---- region sharding over the GPUs of one box ---------------------------------------------------------------------------
struct Shard {
    int gpu;
    uint64_t beg, end;   // half-open site range
};
// Contiguous shards, cut at multiples of `step` (the reference's 100-kb task length, basetype_caller.cpp:474) from
// reg_beg, sizes differing by at most one step; fewer shards than GPUs when the region is short.
std::vector<Shard> shard_region(uint64_t reg_beg, uint64_t reg_end, int n_gpus, uint64_t step = 100000);

// fill(site0, n, packer): add sites [site0, site0+n) to the (cleared) packer, in order.
using TileSource = std::function<void(uint64_t site0, uint32_t n_sites, TilePacker& into)>;
// sink(site0, records, n): called on the calling thread, in coordinate order over the whole region.
using RecordSink = std::function<void(uint64_t site0, const bv_site_out* recs, uint32_t n_sites)>;

struct RunOptions {
    float min_af = 0.01f;
    uint32_t n_samples = 0;
    uint32_t tile_sites = 16384;
    uint32_t n_slots = 2;
    int em_abs_mode = BV_EM_ABS_INT_TRUNC;
    std::vector<int> devices;   // device of shard i is devices[i % devices.size()]; empty: all visible devices
    int n_shards = 0;           // 0: one shard per device
};
// One host worker thread and one context per shard; tiles are packed while the previous one is on the device.
// No inter-GPU communication: shards are independent, the merge is the concatenation in coordinate order.
void run_region(uint64_t reg_beg, uint64_t reg_end, const RunOptions& opt, const TileSource& fill, const RecordSink& sink);

}  // namespace bvhost
