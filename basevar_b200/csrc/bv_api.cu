// bv_api.cu -- kernels' __global__ entry points and the C ABI of include/basevar_b200.h.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -shared -Xcompiler -fPIC
// (see basevar_b200/build.py).  No torch types, no CPU fallback: every entry point that computes needs a
// CUDA device and fails with BV_ERR_CUDA otherwise.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <new>

#include <nvtx3/nvToolsExt.h>   // header-only; a no-op unless a profiler injects itself

#include "../../include/basevar_b200.h"
#include "bv_count_kernel.cuh"
#include "bv_finish_kernels.cuh"
#include "bv_em_kernels.cuh"
#include "bv_call_kernels.cuh"
#include "bv_list_kernel.cuh"
#include "bv_expand_kernel.cuh"
#include "bv_synth.cuh"

constexpr uint32_t kScalarCtasPerSm = 2;      // grid cap of K2, per SM (98 registers: two CTAs resident)
constexpr uint32_t kFisherCtasPerSm = 8;      // grid cap of bv_fisher_kernel, per SM
constexpr uint32_t kMaxTileSites = 1u << 22;  // sites of one tile at most (EM header indices have 28 bits)
static_assert((uint64_t)bv::kMaxBins * kMaxTileSites < (1ull << 31), "EM bin pool offsets of a tile fit 31 bits");

// NVTX range over a scope (SURVEY.md section 5, "Tracing"): nsys / ncu timelines show the host side of every tile
// (submit, wait) and the launch sequence K0, K1, K2, K3, K4a, K4b, K5, K6 under these names.
struct BvRange {
    explicit BvRange(const char* name) { nvtxRangePushA(name); }
    ~BvRange() { nvtxRangePop(); }
    BvRange(const BvRange&) = delete;
    BvRange& operator=(const BvRange&) = delete;
};

namespace bv {

// ======================================================================================================
// Synthetic pileup generator: one thread writes one 16-cell vector of each plane.
// ======================================================================================================
__global__ void __launch_bounds__(256) bv_synth_kernel(const bv_synth_model* __restrict__ model, uint64_t site0,
                                                      uint32_t n_sites, uint32_t n_samples, uint64_t pitch,
                                                      uint8_t* base, uint8_t* qual, uint8_t* strand, uint8_t* mapq,
                                                      uint8_t* ref_base) {
    const uint32_t vec_per_row = (uint32_t)(pitch >> 4);
    const uint64_t n_units = (uint64_t)n_sites * vec_per_row;
    for (uint64_t u = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; u < n_units;
         u += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t s = (uint32_t)(u / vec_per_row);
        const uint32_t v = (uint32_t)(u - (uint64_t)s * vec_per_row);
        const SynthSite ss = synth_site(model, site0 + s);
        if (v == 0) ref_base[s] = "ACGT"[ss.ref];
        uint32_t wb[4], wq[4], wst[4], wm[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            uint32_t xb = 0, xq = 0, xs = 0, xm = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t i = v * 16 + w * 4 + k;
                SynthCell c;
                if (i < n_samples) c = synth_cell(model, ss, i);
                else { c.base = BV_BASE_N; c.qual = 0; c.strand = BV_STRAND_NONE; c.mapq = 0; }
                xb |= (uint32_t)c.base << (8 * k);
                xq |= (uint32_t)c.qual << (8 * k);
                xs |= (uint32_t)c.strand << (8 * k);
                xm |= (uint32_t)c.mapq << (8 * k);
            }
            wb[w] = xb; wq[w] = xq; wst[w] = xs; wm[w] = xm;
        }
        const size_t off = (size_t)s * pitch + (size_t)v * 16;
        *reinterpret_cast<uint4*>(base + off) = make_uint4(wb[0], wb[1], wb[2], wb[3]);
        *reinterpret_cast<uint4*>(qual + off) = make_uint4(wq[0], wq[1], wq[2], wq[3]);
        *reinterpret_cast<uint4*>(strand + off) = make_uint4(wst[0], wst[1], wst[2], wst[3]);
        if (mapq) *reinterpret_cast<uint4*>(mapq + off) = make_uint4(wm[0], wm[1], wm[2], wm[3]);
    }
}

__global__ void __launch_bounds__(256) bv_synth_rpr_kernel(const bv_synth_model* __restrict__ model, uint64_t site0,
                                                          uint32_t n_sites, uint32_t n_samples, uint64_t rpr_pitch,
                                                          uint16_t* rpr) {
    const uint32_t vec_per_row = (uint32_t)(rpr_pitch >> 3);   // 8 cells (16 bytes) per thread
    const uint64_t n_units = (uint64_t)n_sites * vec_per_row;
    for (uint64_t u = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; u < n_units;
         u += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t s = (uint32_t)(u / vec_per_row);
        const uint32_t v = (uint32_t)(u - (uint64_t)s * vec_per_row);
        const SynthSite ss = synth_site(model, site0 + s);
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t i = v * 8 + 2 * k;
            const uint32_t lo = i < n_samples ? synth_rpr(model, ss, i) : 0u;
            const uint32_t hi = i + 1 < n_samples ? synth_rpr(model, ss, i + 1) : 0u;
            w[k] = lo | (hi << 16);
        }
        *reinterpret_cast<uint4*>(rpr + (size_t)s * rpr_pitch + (size_t)v * 8) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

}  // namespace bv

// ======================================================================================================
// Context
// ======================================================================================================
// Scratch of one in-flight tile: work lists and counters (K1 -> K2 -> K3 -> K4) and the EM kernel's spill space.
// Kernels of different tiles may overlap, so every slot (and the device-resident path) owns one.
struct bv_scratch {
    uint32_t* d_lists = nullptr;      // 6 x cap site indices (list_fisher takes two)
    uint32_t* d_counters = nullptr;   // kNumCounters x u32
    uint32_t* d_bin_spill = nullptr;
    double* d_lml_spill = nullptr;
    // K4a -> K4b -> K4c: headers of the EM sites, pool of their bins, EM tasks and their results (bv_em_kernels.cuh)
    bv::EmSiteHdr* d_em_hdr = nullptr;
    uint32_t* d_em_pool = nullptr;
    uint32_t* d_em_tasks = nullptr;
    double* d_em_res = nullptr;
    double* d_em_single = nullptr;    // [cap][4] log-likelihoods of the single-allele models of the EM sites (K4a -> K4b)
    uint32_t em_task_cap[3] = {0, 0, 0};
    uint32_t cap = 0;
};

struct bv_slot {
    cudaStream_t stream = nullptr;
    bv_scratch scratch;
    uint8_t* d_planes = nullptr;   // base | qual | strand, each max_sites * pitch_cap
    uint8_t* d_ref = nullptr;
    bv_site_out* d_out = nullptr;
    bv_site_out* h_out = nullptr;  // pinned
    uint32_t n_sites = 0;
    bool busy = false;
    const uint8_t* qual_host = nullptr;   // this tile's qual plane is read in place from pinned host memory
    size_t h2d_bytes = 0;                 // bytes uploaded for this tile by cudaMemcpyAsync
    // called sites (bv_tile_submit_calls): the kernels write straight into pinned host memory
    bv_call_out* h_calls = nullptr;       // [max_sites]
    bv_group_out* h_groups = nullptr;     // [max_sites * n_groups], allocated by bv_set_groups
    uint32_t* h_counters = nullptr;       // copy of the scratch counters (kCntCalled = number of calls)
    uint8_t* d_aux = nullptr;             // mapq | rpr planes of pageable host tiles (allocated on first use)
    bool with_calls = false;
    // per-site candidate lists (bv_tile_submit_lists / bv_tile_submit_sparse_lists): allocated on first use
    uint32_t* h_lists = nullptr;          // [2 * max_sites] pinned staging of the tile's lists: one word per site, or with
                                          // compact results {site, list word} per listed site
    uint32_t* d_lists = nullptr;          // [2 * max_sites]
    bv_lrt_out* d_lrt = nullptr;          // [max_sites]
    bv_lrt_out* h_lrt = nullptr;          // [max_sites] pinned
    bool with_lists = false;
    bool lists_packed = false;            // h_lrt holds n_listed entries, one per site with a non-empty list, in site order
    uint32_t n_listed = 0;
    // sparse tiles (bv_tile_submit_sparse): the covered cells as uploaded, expanded into d_planes by K0
    uint32_t* d_cells = nullptr;          // [cells_cap] cells, then [cells_cap] aux words
    uint32_t* d_site_start = nullptr;     // [max_sites + 1]
    uint64_t cells_cap = 0;
    bool sparse = false;
    bool out_direct = false;              // the D2H copy went straight into the caller's pinned buffer
    bv_site_out* out_user = nullptr;      // bv_sparse_tile::out
    // compact record transport (BV_OUT_COMPACT)
    bool compact = false;
    const uint8_t* h_ref = nullptr;       // the tile's REF bases (host memory of the caller, valid until the wait)
    uint2* d_brief = nullptr;             // [max_sites]
    bv_site_brief* h_brief = nullptr;     // [max_sites] pinned
    // BASEVAR_B200_TRACE=1: the tile's timeline on its stream (upload begins / ends, kernels end, results are back)
    cudaEvent_t ev_up = nullptr;          // this tile's upload is complete (recorded on the context's copy stream)
    cudaEvent_t ev_trace[4] = {nullptr, nullptr, nullptr, nullptr};
    uint64_t tile_no = 0;
    double t_submit = 0;                  // host clock at submit, seconds since the context's first traced submit
};

struct bv_ctx {
    int device = 0;
    int num_sms = 0;
    bv_params prm{};
    char err[512] = {0};
    double* d_lut = nullptr;
    double* d_logfact = nullptr;
    bv_synth_model* d_model = nullptr;
    bv_scratch dev_scratch;           // bv_tile_run_device
    uint64_t h2d_bytes_total = 0;
    bool profiling = false;
    cudaEvent_t ev[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int task_ctas_per_sm = bv::kTaskLoCtas;      // resident CTAs per SM of bv_em_task_kernel<kTaskLoCtas> (asked of the runtime in bv_create) ...
    int task_ctas_per_sm_hi = bv::kTaskHiCtas;   // ... and of bv_em_task_kernel<kTaskHiCtas>, the build for tiles with many EM tasks
    bool ev_valid = false;
    bool has_model = false;
    uint64_t pitch_cap = 0;
    bv_slot* slots = nullptr;
    uint64_t launches = 0;
    uint8_t* d_group = nullptr;       // [round16(max_samples)] sample -> population group
    uint32_t n_groups = 0;
    cudaEvent_t ev_call[3] = {nullptr, nullptr, nullptr};
    bool ev_call_valid = false;
    cudaEvent_t ev_list[2] = {nullptr, nullptr};   // around K8 bv_list_kernel
    bool ev_list_valid = false;
    bool list_kernel_ready = false;   // bv_list_kernel's shared-memory attribute is set (first lists tile)
    bool list_packed_ready = false;   // the same for bv_list_packed_kernel (first sparse lists tile with compact results)
    // free-standing rank-sum tests (bv_ranksum_test): stream and device scratch made on first use, grown only
    cudaStream_t rs_stream = nullptr;
    uint8_t* d_rs_bases = nullptr;    // [rs_entries_cap]
    int32_t* d_rs_values = nullptr;   // [rs_entries_cap]
    uint64_t* d_rs_start = nullptr;   // [rs_problems_cap + 1]
    uint8_t* d_rs_ref = nullptr;      // [rs_problems_cap] REF characters, then [rs_problems_cap] ALT masks
    double* d_rs_out = nullptr;       // [rs_problems_cap]
    uint64_t rs_entries_cap = 0;
    uint32_t rs_problems_cap = 0;
    cudaEvent_t ev_rs[2] = {nullptr, nullptr};   // around K9 bv_ranksum_test_kernel
    bool ev_rs_valid = false;
    cudaStream_t copy_stream = nullptr;   // uploads of sparse host tiles, in submit order (see upload_sparse)
    bool trace = false;               // BASEVAR_B200_TRACE=1: one line per sparse host tile on stderr at its wait
    cudaEvent_t ev_trace0 = nullptr;  // recorded at the first traced submit: the origin of the timeline
    uint64_t tiles_traced = 0;
    double t_trace0 = 0;
};

static char g_err[512] = "";

static double host_seconds() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

static int set_err(bv_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    snprintf(g_err, sizeof(g_err), "%s", buf);
    if (ctx) snprintf(ctx->err, sizeof(ctx->err), "%s", buf);
    return code;
}

#define BV_CUDA(ctx, call)                                                                              \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return set_err(ctx, BV_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),    \
                           __FILE__, __LINE__);                                                         \
    } while (0)

static void scratch_free(bv_scratch& sc) {
    cudaFree(sc.d_lists); cudaFree(sc.d_counters); cudaFree(sc.d_bin_spill); cudaFree(sc.d_lml_spill);
    cudaFree(sc.d_em_hdr); cudaFree(sc.d_em_pool); cudaFree(sc.d_em_tasks); cudaFree(sc.d_em_res); cudaFree(sc.d_em_single);
    sc = bv_scratch();
}

// make room for tiles of up to n_sites sites (grows only; cudaMalloc synchronises, so slots are sized at bv_create)
static int scratch_reserve(bv_ctx* ctx, bv_scratch& sc, uint32_t n_sites) {
    if (!sc.d_counters) {
        const size_t warps = (size_t)ctx->num_sms * bv::kQualWarps;
        BV_CUDA(ctx, cudaMalloc(&sc.d_counters, bv::kNumCounters * sizeof(uint32_t)));
        BV_CUDA(ctx, cudaMalloc(&sc.d_bin_spill, warps * bv::kMaxBins * sizeof(uint32_t)));
        BV_CUDA(ctx, cudaMalloc(&sc.d_lml_spill, warps * bv::kMaxBins * sizeof(double)));
    }
    if (n_sites > sc.cap) {
        if (sc.d_lists) BV_CUDA(ctx, cudaFree(sc.d_lists));
        sc.d_lists = nullptr;
        sc.cap = 0;
        BV_CUDA(ctx, cudaMalloc(&sc.d_lists, 6 * (size_t)n_sites * sizeof(uint32_t)));
        // EM scratch: room for every site of a tile to be an EM site with kMaxBins bins and all 11 tasks (6, 4 and 1 over subsets
        // of 2, 3 and 4 alleles), so that K4a's allocations cannot fail and every EM site is decided by K4b (bv_em_kernels.cuh):
        // 2,940 bytes per site and slot -- pool 1,920, task results 880, header 64, single-allele log-likelihoods 32, task
        // list 44.  No tile has more than kMaxTileSites sites.
        cudaFree(sc.d_em_hdr); cudaFree(sc.d_em_pool); cudaFree(sc.d_em_tasks); cudaFree(sc.d_em_res); cudaFree(sc.d_em_single);
        sc.d_em_hdr = nullptr; sc.d_em_pool = nullptr; sc.d_em_tasks = nullptr; sc.d_em_res = nullptr; sc.d_em_single = nullptr;
        cudaGetLastError();
        const uint32_t em_sites = n_sites < kMaxTileSites ? n_sites : kMaxTileSites;
        sc.em_task_cap[0] = 6u * em_sites; sc.em_task_cap[1] = 4u * em_sites; sc.em_task_cap[2] = em_sites;
        const size_t n_task = (size_t)11 * em_sites;
        BV_CUDA(ctx, cudaMalloc(&sc.d_em_hdr, (size_t)em_sites * sizeof(bv::EmSiteHdr)));
        BV_CUDA(ctx, cudaMalloc(&sc.d_em_pool, (size_t)em_sites * bv::kMaxBins * sizeof(uint32_t)));
        BV_CUDA(ctx, cudaMalloc(&sc.d_em_tasks, n_task * sizeof(uint32_t)));
        BV_CUDA(ctx, cudaMalloc(&sc.d_em_res, n_task * bv::kEmResDoubles * sizeof(double)));
        BV_CUDA(ctx, cudaMalloc(&sc.d_em_single, (size_t)em_sites * 4 * sizeof(double)));
        sc.cap = n_sites;
    }
    return BV_OK;
}

static int fill_kernel_args(bv_ctx* ctx, const bv_tile* t, bv_site_out* d_out, bv_scratch& sc, bv::SiteKernelArgs* a) {
    if (!t || !t->base || !t->qual || !t->strand || !t->ref_base || !d_out)
        return set_err(ctx, BV_ERR_ARG, "bv_tile: null pointer");
    if (t->pitch % 16 != 0 || t->pitch < t->n_samples)
        return set_err(ctx, BV_ERR_ARG, "bv_tile: pitch %llu must be a multiple of 16 and >= n_samples %u",
                       (unsigned long long)t->pitch, t->n_samples);
    if (t->n_samples > ctx->prm.max_samples)
        return set_err(ctx, BV_ERR_ARG, "bv_tile: n_samples %u > max_samples %u", t->n_samples, ctx->prm.max_samples);
    if (t->n_sites > kMaxTileSites) return set_err(ctx, BV_ERR_ARG, "bv_tile: more than 2^22 sites in one tile");
    if ((((uintptr_t)t->base) | ((uintptr_t)t->qual) | ((uintptr_t)t->strand)) & 15)
        return set_err(ctx, BV_ERR_ARG, "bv_tile: plane pointers must be 16-byte aligned");
    a->base = t->base; a->qual = t->qual; a->strand = t->strand; a->ref_base = t->ref_base;
    a->out = d_out;
    a->lut = ctx->d_lut;
    a->logtab = reinterpret_cast<const double2*>(ctx->d_lut + 4 * bv::kQStride);
    a->logfact = ctx->d_logfact;
    {
        int rc = scratch_reserve(ctx, sc, t->n_sites);
        if (rc != BV_OK) return rc;
    }
    a->bin_spill = sc.d_bin_spill;
    a->lml_spill = sc.d_lml_spill;
    a->list_slow = sc.d_lists;
    a->list_bound = sc.d_lists + sc.cap;
    a->list_em = sc.d_lists + 2 * (size_t)sc.cap;
    a->list_fisher = sc.d_lists + 4 * (size_t)sc.cap;   // [2 * n_sites] of its 2 * cap words
    a->counters = sc.d_counters;
    a->em_hdr = sc.d_em_hdr; a->em_pool = sc.d_em_pool; a->em_tasks = sc.d_em_tasks; a->em_res = sc.d_em_res; a->em_single = sc.d_em_single;
    for (int k = 0; k < 3; ++k) a->em_task_cap[k] = sc.em_task_cap[k];
    a->brief = nullptr; a->full_out = nullptr;   // set by the submit paths of compact tiles
    a->em_resume = 0;
    a->em_task_split = (uint32_t)ctx->num_sms * (uint32_t)ctx->task_ctas_per_sm_hi * (uint32_t)bv::kTaskThreads;   // one round of resident threads
    a->list_called = nullptr;   // set_call_args() turns the called-site kernels on
    a->mapq = nullptr; a->rpr = nullptr; a->aux_pitch = 0; a->rpr_pitch = 0;
    a->sample_group = nullptr; a->calls = nullptr; a->groups = nullptr; a->n_groups = 0; a->pad0 = 0;
    a->pitch = t->pitch;
    a->qual_pitch = t->pitch;
    a->n_sites = t->n_sites;
    a->n_samples = t->n_samples;
    a->min_af = (double)ctx->prm.min_af;     // float -> double: src/basetype_caller.cpp:122,506
    a->em_eps = (double)ctx->prm.em_eps;     // const float epsilon: src/algorithm.h:213
    a->lrt_threshold = (double)ctx->prm.lrt_threshold;
    a->em_max_iter = ctx->prm.em_max_iter;
    a->abs_mode = ctx->prm.em_abs_mode;
    return BV_OK;
}

// Called-site kernels on: K4 lists the called sites, K5 (rank sums) and K6 (population groups) follow.
static int set_call_args(bv_ctx* ctx, const bv_tile* t, const bv_tile_aux* aux, bv_scratch& sc, bv_call_out* calls,
                         bv_group_out* groups, bv::SiteKernelArgs* a) {
    if (!aux || !aux->mapq || !aux->rpr || !calls) return set_err(ctx, BV_ERR_ARG, "bv_tile_aux: null pointer");
    if (aux->rpr_pitch % 8 != 0 || aux->rpr_pitch < t->n_samples)
        return set_err(ctx, BV_ERR_ARG, "bv_tile_aux: rpr_pitch %llu must be a multiple of 8 and >= n_samples %u",
                       (unsigned long long)aux->rpr_pitch, t->n_samples);
    if ((((uintptr_t)aux->mapq) | ((uintptr_t)aux->rpr)) & 15)
        return set_err(ctx, BV_ERR_ARG, "bv_tile_aux: plane pointers must be 16-byte aligned");
    if (ctx->n_groups && !groups) return set_err(ctx, BV_ERR_ARG, "population groups are set but the group output is null");
    a->list_called = sc.d_lists + 3 * (size_t)sc.cap;
    a->mapq = aux->mapq; a->rpr = aux->rpr;
    a->aux_pitch = t->pitch; a->rpr_pitch = aux->rpr_pitch;
    a->sample_group = ctx->d_group;
    a->calls = calls; a->groups = groups;
    a->n_groups = ctx->n_groups;
    return BV_OK;
}

// K2..KF of launch_site_kernel.  pdl: K3..KF with programmatic stream serialization (griddepcontrol, see bv_common.cuh):
// the kernel is launched once every CTA of the kernel before it has triggered, which each does when it has no work left,
// and its CTAs run their prologue (shared-memory tables from constant inputs) on the SMs that kernel has left, while its
// last CTAs finish; their reads of its results wait in grid_dep_wait for its completion.  That takes the launch gap
// (1-2 us) and the prologue off the critical path of every link of the chain.  No deadlock: the dependents are released
// only when every CTA of the primary has triggered or exited, i.e. is resident or gone, so a waiting dependent CTA never
// holds resources that a primary CTA still needs in order to start, even where the primary takes more than one wave.
// Measured on a B200 (profiles/r06_bench_ab.json), two choices:
//   * triggering on the kernels' first lines was slower (C2 step +0.019 ms): the dependents' CTAs then sat waiting on the
//     SMs for the whole of the primary, and K4b's idle build for the whole of the working one;
//   * K2 is launched plainly: chained behind K1 its CTAs land on the SMs in the order K1's CTAs finish, two per SM, and
//     it ran 8 us longer than it does behind a drained K1.
// Profiled tiles launch every kernel without the attribute, with the events between them: per-kernel times of a
// serialised chain, comparable over the history of the project.
static cudaError_t launch_chained(bool pdl, void (*kernel)(bv::SiteKernelArgs), uint32_t grid, uint32_t block, size_t smem,
                                  cudaStream_t stream, const bv::SiteKernelArgs& a) {
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, a);
}

// The basetype core of one tile: K1 (counts, every cell), K2 (scalar finish, one thread per site), K3 / K4 (sites whose
// result depends on base qualities: likelihood-ratio bound, then EM + LRT).  Stream ordered; see csrc/bv_common.cuh.
static int launch_site_kernel(bv_ctx* ctx, const bv::SiteKernelArgs& a, cudaStream_t stream, bool counters_zeroed = false) {
    BvRange range("bv: launch K1 count, K2 scalar, K3 bound, K4a hist, K4b em_task (+ K5 ranksum, K6 group)");
    if (a.n_sites == 0) return BV_OK;
    if (a.n_samples == 0) {   // no cells: every record is all-zero
        BV_CUDA(ctx, cudaMemsetAsync(a.out, 0, (size_t)a.n_sites * sizeof(bv_site_out), stream));
        if (a.brief) BV_CUDA(ctx, cudaMemsetAsync(a.brief, 0, (size_t)a.n_sites * sizeof(uint2), stream));
        return BV_OK;
    }
    if (!counters_zeroed) BV_CUDA(ctx, cudaMemsetAsync(a.counters, 0, bv::kNumCounters * sizeof(uint32_t), stream));
    const bool prof = ctx->profiling;
    if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev[0], stream));
    // K1, persistent: one CTA per SM, each warp strides over the sites; kernel shape by row length
    uint32_t grid;
    if (a.n_samples > (uint32_t)bv::kLongRowSamples) {
        grid = (a.n_sites + bv::kCountWarpsLong - 1) / bv::kCountWarpsLong;
        if (grid > (uint32_t)ctx->num_sms) grid = (uint32_t)ctx->num_sms;
        bv::bv_count_kernel<bv::kCountWarpsLong, bv::kCountStagesLong><<<grid, bv::kCountWarpsLong * 32,
            bv::count_smem_bytes<bv::kCountWarpsLong, bv::kCountStagesLong>(), stream>>>(a);
    } else {
        grid = (a.n_sites + bv::kCountWarpsShort - 1) / bv::kCountWarpsShort;
        if (grid > (uint32_t)ctx->num_sms) grid = (uint32_t)ctx->num_sms;
        bv::bv_count_kernel<bv::kCountWarpsShort, bv::kCountStagesShort><<<grid, bv::kCountWarpsShort * 32,
            bv::count_smem_bytes<bv::kCountWarpsShort, bv::kCountStagesShort>(), stream>>>(a);
    }
    BV_CUDA(ctx, cudaGetLastError());
    if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev[1], stream));
    // K1 and K2 are launched plainly: K1 stays behind the counter memset and the previous tile's KF.  K3..KF are chained.
    const bool pdl = !prof;
    grid = (a.n_sites + bv::kScalarThreads - 1) / bv::kScalarThreads;   // CTAs split K1's work list into equal slices
    if (grid > (uint32_t)ctx->num_sms * kScalarCtasPerSm) grid = (uint32_t)ctx->num_sms * kScalarCtasPerSm;
    BV_CUDA(ctx, launch_chained(false, bv::bv_scalar_kernel, grid, bv::kScalarThreads, 0, stream, a));
    if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev[2], stream));
    // K3 and K4, persistent: each warp strides over groups of 32 sites
    grid = ((a.n_sites + 31) / 32 + bv::kBoundWarps - 1) / bv::kBoundWarps;
    if (grid > (uint32_t)ctx->num_sms) grid = (uint32_t)ctx->num_sms;
    BV_CUDA(ctx, launch_chained(pdl, bv::bv_bound_kernel, grid, bv::kBoundWarps * 32, bv::kBoundSmemBytes, stream, a));
    if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev[3], stream));
    // K4a: one warp per site of the EM list, whose length the host does not know: up to every site of the tile (deep pileups
    // with a small min_af: half of the sites of a 100,000-sample tile), so the grid covers that; warps without work leave at once
    if (a.n_samples > (uint32_t)bv::kLongRowSamples) {
        grid = (a.n_sites + bv::kLongWarps - 1) / bv::kLongWarps;
        if (grid > (uint32_t)ctx->num_sms) grid = (uint32_t)ctx->num_sms;
        BV_CUDA(ctx, launch_chained(pdl, bv::bv_hist_kernel<true>, grid, bv::kLongWarps * 32, bv::kHistLongSmemBytes, stream, a));
    } else {
        grid = (a.n_sites + bv::kQualWarps - 1) / bv::kQualWarps;
        if (grid > (uint32_t)ctx->num_sms) grid = (uint32_t)ctx->num_sms;
        BV_CUDA(ctx, launch_chained(pdl, bv::bv_hist_kernel<false>, grid, bv::kQualWarps * 32, bv::kQualSmemBytes, stream, a));
    }
    if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev[4], stream));
    // K4b: groups of lanes per EM task, CTAs stride over the task lists (their lengths are only known on the device, where the
    // kernel picks the group size from them): always the grid that fills the GPU, CTAs without work leave at once
    grid = (uint32_t)ctx->num_sms * (uint32_t)ctx->task_ctas_per_sm;
    const uint32_t grid_hi = (uint32_t)ctx->num_sms * (uint32_t)ctx->task_ctas_per_sm_hi;
    bv::SiteKernelArgs b = a;
    if (a.abs_mode != BV_EM_ABS_INT_TRUNC) {
        // fabs in the convergence test: EMs of very different lengths; their iterations run with the lanes fed task by task
        // (bv_em_iter_kernel), the rest of every task -- log-likelihood sums, decisions -- from the frequencies that leaves
        BV_CUDA(ctx, launch_chained(pdl, bv::bv_em_iter_kernel, grid, bv::kTaskThreads, bv::kTaskSmemBytes, stream, a));
        ctx->launches += 1;
        b.em_resume = 1;
    }
    // two builds of the kernel (registers / occupancy); the tile's task count decides on the device which of them works
    BV_CUDA(ctx, launch_chained(pdl, bv::bv_em_task_kernel<bv::kTaskLoCtas>, grid, bv::kTaskThreads, bv::kTaskSmemBytes, stream, b));
    BV_CUDA(ctx, launch_chained(pdl, bv::bv_em_task_kernel<bv::kTaskHiCtas>, grid_hi, bv::kTaskThreads, bv::kTaskSmemBytes, stream, b));
    ctx->launches += 1;
    if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev[5], stream));
    // the Fisher tests K2 and K4 listed (as many as two per site; the counts are on the device): grid-stride
    grid = (4u * a.n_sites + bv::kFisherThreads - 1) / bv::kFisherThreads;   // (a pair of lanes per test)
    if (grid > (uint32_t)ctx->num_sms * kFisherCtasPerSm) grid = (uint32_t)ctx->num_sms * kFisherCtasPerSm;
    BV_CUDA(ctx, launch_chained(pdl, bv::bv_fisher_kernel, grid, bv::kFisherThreads, 0, stream, a));
    if (prof) { BV_CUDA(ctx, cudaEventRecord(ctx->ev[6], stream)); ctx->ev_valid = true; }
    ctx->launches += 6;
    if (a.list_called) {
        // K5 / K6: the called sites (a few per mille of the tile at 0.1x); grids sized for the worst case, warps
        // without work leave at once
        if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev_call[0], stream));
        grid = (a.n_sites + bv::kCallWarps - 1) / bv::kCallWarps;
        if (grid > (uint32_t)ctx->num_sms) grid = (uint32_t)ctx->num_sms;
        bv::bv_ranksum_kernel<<<grid, bv::kCallWarps * 32, bv::kCallSmemBytes, stream>>>(a);
        BV_CUDA(ctx, cudaGetLastError());
        ctx->launches += 1;
        if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev_call[1], stream));
        if (a.n_groups) {
            grid = (a.n_sites + bv::kQualWarps - 1) / bv::kQualWarps;
            if (grid > (uint32_t)ctx->num_sms) grid = (uint32_t)ctx->num_sms;
            bv::bv_group_kernel<<<grid, bv::kQualWarps * 32, bv::kQualSmemBytes, stream>>>(a);
            BV_CUDA(ctx, cudaGetLastError());
            ctx->launches += 1;
        }
        if (prof) { BV_CUDA(ctx, cudaEventRecord(ctx->ev_call[2], stream)); ctx->ev_call_valid = true; }
    }
    return BV_OK;
}

// K8 after the standard kernels of the tile (it reads their records), one warp per listed site: over the n = n_sites words of
// d_lists (bv_list_kernel), or over the n {site, list word} pairs of a compact tile's packed list, entry k for pair k
// (bv_list_packed_kernel, d_pairs).
static int launch_list_kernel(bv_ctx* ctx, const bv::SiteKernelArgs& a, const uint32_t* d_lists, const uint2* d_pairs, uint32_t n,
                              bv_lrt_out* d_lrt, cudaStream_t stream) {
    BvRange range(d_pairs ? "bv: launch K8 list (packed)" : "bv: launch K8 list");
    if (n == 0) return BV_OK;
    if (a.n_samples == 0) {   // no reads anywhere: every entry is all-zero
        BV_CUDA(ctx, cudaMemsetAsync(d_lrt, 0, (size_t)n * sizeof(bv_lrt_out), stream));
        return BV_OK;
    }
    // on first use: a context that never runs K8 loads and sets up exactly what it did without it
    bool& ready = d_pairs ? ctx->list_packed_ready : ctx->list_kernel_ready;
    if (!ready) {
        BV_CUDA(ctx, cudaFuncSetAttribute(d_pairs ? (const void*)bv::bv_list_packed_kernel : (const void*)bv::bv_list_kernel,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kQualSmemBytes));
        ready = true;
    }
    const bool prof = ctx->profiling;
    if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev_list[0], stream));
    uint32_t grid = (n + bv::kQualWarps - 1) / bv::kQualWarps;
    if (grid > (uint32_t)ctx->num_sms) grid = (uint32_t)ctx->num_sms;   // (the bin spill rows are sized for this grid)
    if (d_pairs) bv::bv_list_packed_kernel<<<grid, bv::kQualWarps * 32, bv::kQualSmemBytes, stream>>>(a, d_pairs, n, d_lrt);
    else bv::bv_list_kernel<<<grid, bv::kQualWarps * 32, bv::kQualSmemBytes, stream>>>(a, d_lists, d_lrt);
    BV_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    if (prof) { BV_CUDA(ctx, cudaEventRecord(ctx->ev_list[1], stream)); ctx->ev_list_valid = true; }
    return BV_OK;
}

// The slot's list staging and results, allocated on the first lists tile.
static int lists_reserve(bv_ctx* ctx, bv_slot& s) {
    if (s.h_lists) return BV_OK;
    const size_t n = ctx->prm.max_sites;
    BV_CUDA(ctx, cudaHostAlloc(&s.h_lists, 2 * n * sizeof(uint32_t), cudaHostAllocDefault));
    BV_CUDA(ctx, cudaHostAlloc(&s.h_lrt, n * sizeof(bv_lrt_out), cudaHostAllocDefault));
    BV_CUDA(ctx, cudaMalloc(&s.d_lists, 2 * n * sizeof(uint32_t)));
    BV_CUDA(ctx, cudaMalloc(&s.d_lrt, n * sizeof(bv_lrt_out)));
    return BV_OK;
}

// Host check of a tile's lists (what the kernel would otherwise treat as empty): BV_OK or BV_ERR_ARG.
static int check_lists(bv_ctx* ctx, const uint8_t (*lists)[4], uint32_t n_sites) {
    for (uint32_t i = 0; i < n_sites; ++i) {
        uint32_t w, order;
        memcpy(&w, lists[i], 4);
        if (bv::list_decode(w, order) < 0)
            return set_err(ctx, BV_ERR_ARG, "lists[%u] = {%u, %u, %u, %u}: a base repeats or a code is neither 0..3 nor BV_LIST_END", i,
                           lists[i][0], lists[i][1], lists[i][2], lists[i][3]);
    }
    return BV_OK;
}

// The cells of one site, words16 known to have room for the worst case.  The common cell -- ascending, gap < 31, strand + or - --
// is one load, a few shifts and one store; everything else leaves through the slow path of the caller.
template <bool AUX>
static inline const uint32_t* encode16_run(const uint32_t* __restrict__ p, const uint32_t* __restrict__ end, const uint32_t* __restrict__ aux32,
                                           uint16_t* __restrict__& o, uint32_t* __restrict__& oa, uint32_t& next) {
    uint32_t nx = next;
    uint16_t* out = o;
    uint32_t* outa = oa;
    for (; p < end; ++p) {
        const uint32_t w = *p, i = w & (BV_CELL_MAX_SAMPLES - 1u), f12 = w >> 20;   // f12: base | strand << 3 | phred << 5
        uint32_t gap = i - nx;   // i < next wraps to a huge value
        if (__builtin_expect(gap >= BV_CELL16_GAP_SKIP || (f12 & 0x10u), 0)) {
            if ((f12 & 0x10u) || gap >= BV_CELL_MAX_SAMPLES) break;   // a strand without a 16-bit form, or descending samples: the caller reports it
            do {   // one cell in 26 at 0.1x: "skip 31 samples" words in front of it
                *out++ = (uint16_t)BV_CELL16_GAP_SKIP;
                if (AUX) *outa++ = 0;
                gap -= BV_CELL16_GAP_SKIP;
            } while (gap >= BV_CELL16_GAP_SKIP);
        }
        *out++ = (uint16_t)(gap | (((f12 & 0xfu) | ((f12 >> 5) << 4)) << 5));
        if (AUX) *outa++ = aux32 ? aux32[p - end] : 0;   // (aux32 is passed pre-offset so that aux32[p - end] is this cell's word)
        nx = i + 1;
    }
    next = nx; o = out; oa = outa;
    return p;
}

namespace bv {   // bv_encode16.cpp: the same loop, eight cells per step (AVX2, chosen at run time)
bool encode16_have_avx2();
template <bool AUX>
const uint32_t* encode16_run_avx2(const uint32_t* __restrict__ p, const uint32_t* __restrict__ end, const uint32_t* __restrict__ aux32,
                                  uint16_t* __restrict__& o, uint32_t* __restrict__& oa, uint32_t& next);
}  // namespace bv

// The records of a tile on their way back: all of them (BV_OUT_RECORDS), or the briefs plus the full records of the sites that
// need one (BV_OUT_COMPACT; the pack kernel writes those into the slot's pinned list itself).
static int return_records(bv_ctx* ctx, bv_slot& s, const bv::SiteKernelArgs& a, uint32_t n_sites, bv_site_out* dst) {
    if (!n_sites) return BV_OK;
    if (!s.compact) {
        BV_CUDA(ctx, cudaMemcpyAsync(dst, s.d_out, (size_t)n_sites * sizeof(bv_site_out), cudaMemcpyDeviceToHost, s.stream));
        return BV_OK;
    }
    if (a.n_samples) {
        uint32_t grid = (n_sites + 255) / 256;
        if (grid > (uint32_t)ctx->num_sms * 8u) grid = (uint32_t)ctx->num_sms * 8u;
        bv::bv_pack_kernel<<<grid, 256, 0, s.stream>>>(a);
        BV_CUDA(ctx, cudaGetLastError());
        ctx->launches += 1;
    }
    BV_CUDA(ctx, cudaMemcpyAsync(s.h_brief, s.d_brief, (size_t)n_sites * sizeof(uint2), cudaMemcpyDeviceToHost, s.stream));
    return BV_OK;
}

extern "C" {

int bv_version(void) { return BV_VERSION_MAJOR * 1000 + BV_VERSION_MINOR; }

const char* bv_last_error(const bv_ctx* ctx) { return ctx ? ctx->err : g_err; }

uint64_t bv_launch_count(const bv_ctx* ctx) { return ctx ? ctx->launches : 0; }
uint64_t bv_h2d_bytes(const bv_ctx* ctx) { return ctx ? ctx->h2d_bytes_total : 0; }

int bv_set_profiling(bv_ctx* ctx, int on) {
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    if (on && !ctx->ev[0]) {
        for (int i = 0; i < 7; ++i) BV_CUDA(ctx, cudaEventCreate(&ctx->ev[i]));
        for (int i = 0; i < 3; ++i) BV_CUDA(ctx, cudaEventCreate(&ctx->ev_call[i]));
        for (int i = 0; i < 2; ++i) BV_CUDA(ctx, cudaEventCreate(&ctx->ev_list[i]));
        for (int i = 0; i < 2; ++i) BV_CUDA(ctx, cudaEventCreate(&ctx->ev_rs[i]));
    }
    ctx->profiling = on != 0;
    ctx->ev_valid = false;
    ctx->ev_call_valid = false;
    ctx->ev_list_valid = false;
    ctx->ev_rs_valid = false;
    return BV_OK;
}

int bv_last_call_kernel_times(bv_ctx* ctx, float ms[2]) {
    if (!ctx || !ms) return set_err(ctx, BV_ERR_ARG, "null argument");
    if (!ctx->ev_call_valid) return set_err(ctx, BV_ERR_STATE, "no profiled tile with called-site kernels yet");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    BV_CUDA(ctx, cudaEventSynchronize(ctx->ev_call[2]));
    for (int i = 0; i < 2; ++i) BV_CUDA(ctx, cudaEventElapsedTime(&ms[i], ctx->ev_call[i], ctx->ev_call[i + 1]));
    return BV_OK;
}

int bv_last_list_kernel_time(bv_ctx* ctx, float* ms) {
    if (!ctx || !ms) return set_err(ctx, BV_ERR_ARG, "null argument");
    if (!ctx->ev_list_valid) return set_err(ctx, BV_ERR_STATE, "no profiled tile with the list kernel yet");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    BV_CUDA(ctx, cudaEventSynchronize(ctx->ev_list[1]));
    BV_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev_list[0], ctx->ev_list[1]));
    return BV_OK;
}

int bv_last_ranksum_kernel_time(bv_ctx* ctx, float* ms) {
    if (!ctx || !ms) return set_err(ctx, BV_ERR_ARG, "null argument");
    if (!ctx->ev_rs_valid) return set_err(ctx, BV_ERR_STATE, "no profiled bv_ranksum_test call yet");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    BV_CUDA(ctx, cudaEventSynchronize(ctx->ev_rs[1]));
    BV_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev_rs[0], ctx->ev_rs[1]));
    return BV_OK;
}

int bv_last_kernel_times(bv_ctx* ctx, float ms[4]) {
    if (!ctx || !ms) return set_err(ctx, BV_ERR_ARG, "null argument");
    if (!ctx->ev_valid) return set_err(ctx, BV_ERR_STATE, "no profiled tile yet (bv_set_profiling)");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    BV_CUDA(ctx, cudaEventSynchronize(ctx->ev[5]));
    for (int i = 0; i < 3; ++i) BV_CUDA(ctx, cudaEventElapsedTime(&ms[i], ctx->ev[i], ctx->ev[i + 1]));
    BV_CUDA(ctx, cudaEventElapsedTime(&ms[3], ctx->ev[3], ctx->ev[5]));   // K4 = K4a + K4b
    return BV_OK;
}

int bv_last_em_kernel_times(bv_ctx* ctx, float ms[2]) {
    if (!ctx || !ms) return set_err(ctx, BV_ERR_ARG, "null argument");
    if (!ctx->ev_valid) return set_err(ctx, BV_ERR_STATE, "no profiled tile yet (bv_set_profiling)");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    BV_CUDA(ctx, cudaEventSynchronize(ctx->ev[5]));
    for (int i = 0; i < 2; ++i) BV_CUDA(ctx, cudaEventElapsedTime(&ms[i], ctx->ev[3 + i], ctx->ev[4 + i]));
    return BV_OK;
}

int bv_last_fisher_kernel_time(bv_ctx* ctx, float* ms) {
    if (!ctx || !ms) return set_err(ctx, BV_ERR_ARG, "null argument");
    if (!ctx->ev_valid) return set_err(ctx, BV_ERR_STATE, "no profiled tile yet (bv_set_profiling)");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    BV_CUDA(ctx, cudaEventSynchronize(ctx->ev[6]));
    BV_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev[5], ctx->ev[6]));
    return BV_OK;
}

static int upload_tables(bv_ctx* ctx) {
    // per-phred likelihood table: eps = exp((q) * MLN10TO10) with glibc exp, exactly the reference's expression
    // (src/basetype.cpp:47, MLN10TO10 at src/basetype.h:20); 1-eps and eps/3 are single IEEE operations.
    const double MLN10TO10 = -0.23025850929940458;
    double lut[4 * bv::kQStride + 2 * bv::kLogTabEntries];
    for (int q = 0; q < bv::kQStride; ++q) {
        double eps = exp((double)q * MLN10TO10);
        double ome = 1.0 - eps, e3 = eps / 3;
        lut[bv::kLutOneMinusEps * bv::kQStride + q] = ome;
        lut[bv::kLutEpsThird * bv::kQStride + q] = e3;
        lut[bv::kLutLogMatch * bv::kQStride + q] = log(ome);
        lut[bv::kLutLogMis * bv::kQStride + q] = log(e3);
    }
    // log_tab() of bv_em_kernels.cuh: {1 / c rounded, -log of that rounded value}, c = the midpoint of the i-th of 128 mantissa intervals
    for (int i = 0; i < bv::kLogTabEntries; ++i) {
        const double inv = 1.0 / (1.0 + ((double)i + 0.5) / (double)bv::kLogTabEntries);
        lut[4 * bv::kQStride + 2 * i] = inv;
        lut[4 * bv::kQStride + 2 * i + 1] = -(double)logl((long double)inv);
    }
    BV_CUDA(ctx, cudaMalloc(&ctx->d_lut, sizeof(lut)));
    BV_CUDA(ctx, cudaMemcpy(ctx->d_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
    // log-factorials: lgamma(k+1) from glibc, the values lbinom() uses (htslib/kfunc.c:197-201)
    const size_t n = (size_t)ctx->prm.max_samples + 2;
    double* lf = (double*)malloc(n * sizeof(double));
    if (!lf) return set_err(ctx, BV_ERR_NOMEM, "out of host memory");
    for (size_t k = 0; k < n; ++k) lf[k] = lgamma((double)(k + 1));
    cudaError_t e = cudaMalloc(&ctx->d_logfact, n * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(ctx->d_logfact, lf, n * sizeof(double), cudaMemcpyHostToDevice);
    free(lf);
    BV_CUDA(ctx, e);
    return BV_OK;
}

int bv_create(int device, const bv_params* params, bv_ctx** out_ctx) {
    if (!params || !out_ctx) return set_err(nullptr, BV_ERR_ARG, "bv_create: null argument");
    *out_ctx = nullptr;
    if (params->max_samples == 0 || params->max_samples > 2000000u)
        return set_err(nullptr, BV_ERR_ARG, "bv_create: max_samples must be in 1..2000000");
    if (params->n_slots > 64) return set_err(nullptr, BV_ERR_ARG, "bv_create: n_slots > 64");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return set_err(nullptr, BV_ERR_CUDA, "bv_create: no CUDA device (%s); this library has no CPU fallback",
                       cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return set_err(nullptr, BV_ERR_ARG, "bv_create: bad device %d", device);
    bv_ctx* ctx = new (std::nothrow) bv_ctx();
    if (!ctx) return set_err(nullptr, BV_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    ctx->prm = *params;
    int rc = BV_OK;
    do {
        if (cudaSetDevice(device) != cudaSuccess) { rc = set_err(nullptr, BV_ERR_CUDA, "cudaSetDevice failed"); break; }
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { rc = set_err(nullptr, BV_ERR_CUDA, "cudaGetDeviceProperties failed"); break; }
        ctx->num_sms = prop.multiProcessorCount;
        if (cudaFuncSetAttribute(bv::bv_count_kernel<bv::kCountWarpsShort, bv::kCountStagesShort>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)bv::count_smem_bytes<bv::kCountWarpsShort, bv::kCountStagesShort>()) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_count_kernel<bv::kCountWarpsLong, bv::kCountStagesLong>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)bv::count_smem_bytes<bv::kCountWarpsLong, bv::kCountStagesLong>()) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_bound_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kBoundSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_hist_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kQualSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_hist_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kHistLongSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_em_task_kernel<bv::kTaskLoCtas>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kTaskSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_em_task_kernel<bv::kTaskHiCtas>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kTaskSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_em_iter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kTaskSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kQualSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_ranksum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kCallSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_expand_kernel<BV_CELLS_U32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kExpandSmemBytes) != cudaSuccess ||
            cudaFuncSetAttribute(bv::bv_expand_kernel<BV_CELLS_U16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kExpandSmemBytes) != cudaSuccess) {
            rc = set_err(nullptr, BV_ERR_CUDA, "cudaFuncSetAttribute failed: %s (device is not sm_100?)",
                         cudaGetErrorString(cudaGetLastError()));
            break;
        }
        {   // the EM task kernel's grid: what is resident at once (registers / shared memory decide)
            int nb = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, bv::bv_em_task_kernel<bv::kTaskLoCtas>, bv::kTaskThreads, bv::kTaskSmemBytes) == cudaSuccess && nb > 0)
                ctx->task_ctas_per_sm = nb;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, bv::bv_em_task_kernel<bv::kTaskHiCtas>, bv::kTaskThreads, bv::kTaskSmemBytes) == cudaSuccess && nb > 0)
                ctx->task_ctas_per_sm_hi = nb;
            cudaGetLastError();
        }
        {
            const char* z = getenv("BASEVAR_B200_TRACE");
            ctx->trace = z && z[0] == '1';
        }
        rc = upload_tables(ctx);
        if (rc != BV_OK) break;
        ctx->pitch_cap = ((uint64_t)params->max_samples + 15) / 16 * 16;
        if (params->n_slots > 0 && params->max_sites > 0) {
            ctx->slots = new (std::nothrow) bv_slot[params->n_slots];
            if (!ctx->slots) { rc = set_err(nullptr, BV_ERR_NOMEM, "out of host memory"); break; }
            const size_t plane = (size_t)params->max_sites * ctx->pitch_cap;
            if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { rc = set_err(nullptr, BV_ERR_CUDA, "cudaStreamCreate failed"); break; }
            for (uint32_t i = 0; i < params->n_slots && rc == BV_OK; ++i) {
                bv_slot& s = ctx->slots[i];
                cudaError_t ce = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking);
                if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&s.ev_up, cudaEventDisableTiming);
                if (ce == cudaSuccess) ce = cudaMalloc(&s.d_planes, 3 * plane);
                if (ce == cudaSuccess) ce = cudaMalloc(&s.d_ref, params->max_sites);
                if (ce == cudaSuccess) ce = cudaMalloc(&s.d_out, (size_t)params->max_sites * sizeof(bv_site_out));
                // mapped: compact tiles have the device write their full records straight into it
                if (ce == cudaSuccess) ce = cudaHostAlloc(&s.h_out, (size_t)params->max_sites * sizeof(bv_site_out), cudaHostAllocMapped);
                if (ce == cudaSuccess) ce = cudaMalloc(&s.d_brief, (size_t)params->max_sites * sizeof(uint2));
                if (ce == cudaSuccess) ce = cudaHostAlloc(&s.h_brief, (size_t)params->max_sites * sizeof(bv_site_brief), cudaHostAllocDefault);
                if (ce == cudaSuccess) ce = cudaHostAlloc(&s.h_calls, (size_t)params->max_sites * sizeof(bv_call_out), cudaHostAllocMapped);
                if (ce == cudaSuccess) ce = cudaHostAlloc(&s.h_counters, bv::kNumCounters * sizeof(uint32_t), cudaHostAllocDefault);
                if (ce != cudaSuccess) rc = set_err(nullptr, BV_ERR_CUDA, "slot allocation failed: %s", cudaGetErrorString(ce));
                else rc = scratch_reserve(ctx, s.scratch, params->max_sites);
            }
        }
    } while (0);
    if (rc != BV_OK) { bv_destroy(ctx); return rc; }
    *out_ctx = ctx;
    return BV_OK;
}

void bv_destroy(bv_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->slots) {
        for (uint32_t i = 0; i < ctx->prm.n_slots; ++i) {
            bv_slot& s = ctx->slots[i];
            if (s.stream) { cudaStreamSynchronize(s.stream); cudaStreamDestroy(s.stream); }
            cudaFree(s.d_planes); cudaFree(s.d_ref); cudaFree(s.d_out);
            scratch_free(s.scratch);
            if (s.h_out) cudaFreeHost(s.h_out);
            if (s.h_brief) cudaFreeHost(s.h_brief);
            cudaFree(s.d_brief);
            if (s.h_calls) cudaFreeHost(s.h_calls);
            if (s.h_groups) cudaFreeHost(s.h_groups);
            if (s.h_counters) cudaFreeHost(s.h_counters);
            cudaFree(s.d_aux);
            if (s.h_lists) cudaFreeHost(s.h_lists);
            if (s.h_lrt) cudaFreeHost(s.h_lrt);
            cudaFree(s.d_lists); cudaFree(s.d_lrt);
            cudaFree(s.d_cells); cudaFree(s.d_site_start);
            for (int k = 0; k < 4; ++k) if (s.ev_trace[k]) cudaEventDestroy(s.ev_trace[k]);
            if (s.ev_up) cudaEventDestroy(s.ev_up);
        }
        delete[] ctx->slots;
    }
    cudaFree(ctx->d_lut); cudaFree(ctx->d_logfact); cudaFree(ctx->d_model); cudaFree(ctx->d_group);
    scratch_free(ctx->dev_scratch);
    for (int i = 0; i < 7; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < 3; ++i) if (ctx->ev_call[i]) cudaEventDestroy(ctx->ev_call[i]);
    for (int i = 0; i < 2; ++i) if (ctx->ev_list[i]) cudaEventDestroy(ctx->ev_list[i]);
    for (int i = 0; i < 2; ++i) if (ctx->ev_rs[i]) cudaEventDestroy(ctx->ev_rs[i]);
    if (ctx->rs_stream) { cudaStreamSynchronize(ctx->rs_stream); cudaStreamDestroy(ctx->rs_stream); }
    cudaFree(ctx->d_rs_bases); cudaFree(ctx->d_rs_values); cudaFree(ctx->d_rs_start); cudaFree(ctx->d_rs_ref); cudaFree(ctx->d_rs_out);
    if (ctx->ev_trace0) cudaEventDestroy(ctx->ev_trace0);
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    delete ctx;
}

int bv_set_params(bv_ctx* ctx, const bv_params* p) {
    if (!ctx || !p) return set_err(ctx, BV_ERR_ARG, "bv_set_params: null argument");
    ctx->prm.min_af = p->min_af;
    ctx->prm.lrt_threshold = p->lrt_threshold;
    ctx->prm.em_max_iter = p->em_max_iter;
    ctx->prm.em_eps = p->em_eps;
    ctx->prm.em_abs_mode = p->em_abs_mode;
    return BV_OK;
}

// The prologue of the device-resident entry points: the tile's kernel arguments over the context's own scratch.
// no_compact: the entry point refuses BV_OUT_COMPACT (bv_tile_run_device ignores out_mode).
static int device_tile_args(bv_ctx* ctx, const bv_tile* tile, bv_site_out* d_out, bool no_compact, bv::SiteKernelArgs* a) {
    if (no_compact && tile && tile->out_mode == BV_OUT_COMPACT)
        return set_err(ctx, BV_ERR_ARG, "BV_OUT_COMPACT: device-resident tiles have no compact form");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    return fill_kernel_args(ctx, tile, d_out, ctx->dev_scratch, a);
}

int bv_tile_run_device(bv_ctx* ctx, const bv_tile* tile, bv_site_out* d_out, void* stream) {
    BvRange range("bv_tile_run_device");
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    if (tile && tile->location != BV_LOC_DEVICE) return set_err(ctx, BV_ERR_ARG, "bv_tile_run_device: tile must be device resident");
    bv::SiteKernelArgs a;
    int rc = device_tile_args(ctx, tile, d_out, false, &a);
    if (rc != BV_OK) return rc;
    return launch_site_kernel(ctx, a, (cudaStream_t)stream);
}

int bv_tile_run_device_calls(bv_ctx* ctx, const bv_tile* tile, const bv_tile_aux* aux, bv_site_out* d_out,
                             bv_call_out* d_calls, bv_group_out* d_groups, uint32_t* d_n_calls, void* stream) {
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    if (tile && tile->location != BV_LOC_DEVICE) return set_err(ctx, BV_ERR_ARG, "bv_tile_run_device_calls: tile must be device resident");
    if (!d_n_calls) return set_err(ctx, BV_ERR_ARG, "bv_tile_run_device_calls: null d_n_calls");
    bv::SiteKernelArgs a;
    int rc = device_tile_args(ctx, tile, d_out, true, &a);
    if (rc != BV_OK) return rc;
    rc = set_call_args(ctx, tile, aux, ctx->dev_scratch, d_calls, d_groups, &a);
    if (rc != BV_OK) return rc;
    if (a.n_sites == 0 || a.n_samples == 0) {
        BV_CUDA(ctx, cudaMemsetAsync(d_n_calls, 0, sizeof(uint32_t), (cudaStream_t)stream));
        return launch_site_kernel(ctx, a, (cudaStream_t)stream);
    }
    rc = launch_site_kernel(ctx, a, (cudaStream_t)stream);
    if (rc != BV_OK) return rc;
    BV_CUDA(ctx, cudaMemcpyAsync(d_n_calls, a.counters + bv::kCntCalled, sizeof(uint32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return BV_OK;
}

int bv_tile_run_device_lists(bv_ctx* ctx, const bv_tile* tile, const uint8_t (*d_lists)[4], bv_site_out* d_out,
                             bv_lrt_out* d_lrt_out, void* stream) {
    BvRange range("bv_tile_run_device_lists");
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    if (tile && tile->location != BV_LOC_DEVICE) return set_err(ctx, BV_ERR_ARG, "bv_tile_run_device_lists: tile must be device resident");
    if (tile && tile->n_sites && (!d_lists || !d_lrt_out)) return set_err(ctx, BV_ERR_ARG, "bv_tile_run_device_lists: null lists / output");
    if (((uintptr_t)d_lists) & 3) return set_err(ctx, BV_ERR_ARG, "bv_tile_run_device_lists: d_lists must be 4-byte aligned");
    bv::SiteKernelArgs a;
    int rc = device_tile_args(ctx, tile, d_out, true, &a);
    if (rc != BV_OK) return rc;
    rc = launch_site_kernel(ctx, a, (cudaStream_t)stream);
    if (rc != BV_OK) return rc;
    return launch_list_kernel(ctx, a, reinterpret_cast<const uint32_t*>(d_lists), nullptr, a.n_sites, d_lrt_out, (cudaStream_t)stream);
}

int bv_set_groups(bv_ctx* ctx, const uint8_t* sample_group, uint32_t n_samples, uint32_t n_groups) {
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    if (n_groups > BV_MAX_GROUPS) return set_err(ctx, BV_ERR_ARG, "bv_set_groups: more than %d groups", BV_MAX_GROUPS);
    if (n_groups && (!sample_group || n_samples > ctx->prm.max_samples))
        return set_err(ctx, BV_ERR_ARG, "bv_set_groups: bad sample_group / n_samples");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    for (uint32_t i = 0; ctx->slots && i < ctx->prm.n_slots; ++i)
        if (ctx->slots[i].busy) return set_err(ctx, BV_ERR_STATE, "bv_set_groups: slot %u is busy", i);
    for (uint32_t i = 0; ctx->slots && i < ctx->prm.n_slots; ++i) {
        bv_slot& s = ctx->slots[i];
        if (s.h_groups) { BV_CUDA(ctx, cudaFreeHost(s.h_groups)); s.h_groups = nullptr; }
        if (n_groups)
            BV_CUDA(ctx, cudaHostAlloc(&s.h_groups, (size_t)ctx->prm.max_sites * n_groups * sizeof(bv_group_out), cudaHostAllocMapped));
    }
    ctx->n_groups = 0;
    if (n_groups == 0) return BV_OK;
    const size_t padded = ((size_t)ctx->prm.max_samples + 15) / 16 * 16;
    if (!ctx->d_group) BV_CUDA(ctx, cudaMalloc(&ctx->d_group, padded));
    uint8_t* tmp = (uint8_t*)malloc(padded);
    if (!tmp) return set_err(ctx, BV_ERR_NOMEM, "out of host memory");
    memset(tmp, BV_GROUP_NONE, padded);
    for (uint32_t i = 0; i < n_samples; ++i) tmp[i] = sample_group[i] < n_groups ? sample_group[i] : (uint8_t)BV_GROUP_NONE;
    cudaError_t e = cudaMemcpy(ctx->d_group, tmp, padded, cudaMemcpyHostToDevice);
    free(tmp);
    BV_CUDA(ctx, e);
    ctx->n_groups = n_groups;
    return BV_OK;
}

// pinned (or otherwise device-accessible) host memory: the pointer the kernels can use, else null
static const void* host_device_pointer(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) return at.devicePointer;
    cudaGetLastError();   // not registered: a sticky-free error on older runtimes
    return nullptr;
}

// The slot of a submit or a wait; null for a null context or a bad slot index, with the error (BV_ERR_ARG) set.
static bv_slot* slot_of(bv_ctx* ctx, int slot) {
    if (!ctx) { set_err(nullptr, BV_ERR_ARG, "null context"); return nullptr; }
    if (slot < 0 || (uint32_t)slot >= ctx->prm.n_slots || !ctx->slots) { set_err(ctx, BV_ERR_ARG, "bad slot %d", slot); return nullptr; }
    return &ctx->slots[slot];
}

// A tile's lists, checked and staged in the slot's pinned memory before anything is queued (a refused tile leaves the slot as it
// was): one word per site, or for packed results {site, list word} pairs of the sites with a non-empty list, in site order.
static int stage_lists(bv_ctx* ctx, bv_slot& s, const uint8_t (*lists)[4], uint32_t n_sites, bool packed, uint32_t* n_listed) {
    int rc = check_lists(ctx, lists, n_sites);
    if (rc != BV_OK) return rc;
    rc = lists_reserve(ctx, s);
    if (rc != BV_OK) return rc;
    *n_listed = 0;
    if (packed) {
        uint2* pairs = reinterpret_cast<uint2*>(s.h_lists);
        for (uint32_t i = 0; i < n_sites; ++i) {
            if (lists[i][0] == BV_LIST_END) continue;
            uint32_t w;
            memcpy(&w, lists[i], 4);
            pairs[(*n_listed)++] = make_uint2(i, w);
        }
    } else if (n_sites) {
        memcpy(s.h_lists, lists, (size_t)n_sites * sizeof(uint32_t));
    }
    return BV_OK;
}

// Dense tile: the planes of a host tile go up on the slot's stream; a device-resident tile is read where it is.  Fills `a` and
// s.h2d_bytes.
static int upload_dense(bv_ctx* ctx, bv_slot& s, const bv_tile* tile, const bv_tile_aux* aux, bool with_calls, bv::SiteKernelArgs* a) {
    bv_tile dev = *tile;
    if (tile->location == BV_LOC_HOST) {
        if (!tile->base || !tile->qual || !tile->strand || !tile->ref_base) return set_err(ctx, BV_ERR_ARG, "bv_tile: null pointer");
        if (tile->pitch % 16 != 0 || tile->pitch < tile->n_samples || tile->n_samples > ctx->prm.max_samples)
            return set_err(ctx, BV_ERR_ARG, "bv_tile: bad pitch/n_samples");
        // device rows are re-pitched to round16(n_samples) so that no padding crosses PCIe
        const uint64_t dp = ((uint64_t)tile->n_samples + 15) / 16 * 16;
        const size_t plane = (size_t)ctx->prm.max_sites * ctx->pitch_cap;
        uint8_t* d[3] = {s.d_planes, s.d_planes + plane, s.d_planes + 2 * plane};
        const uint8_t* h[3] = {tile->base, tile->qual, tile->strand};
        // The qual plane is read for the minority of rows whose result depends on base qualities (kernels K3 / K4).
        // When it lives in pinned host memory the kernels fetch exactly those rows over PCIe themselves (zero copy),
        // and the plane is not uploaded at all; pageable memory is copied like the other planes.
        const uint8_t* qual_zero_copy = nullptr;
        if (tile->n_sites) qual_zero_copy = static_cast<const uint8_t*>(host_device_pointer(tile->qual));
        for (int k = 0; k < 3 && tile->n_sites; ++k) {
            if (k == 1 && qual_zero_copy) continue;
            if (dp == tile->pitch)
                BV_CUDA(ctx, cudaMemcpyAsync(d[k], h[k], (size_t)tile->n_sites * dp, cudaMemcpyHostToDevice, s.stream));
            else
                BV_CUDA(ctx, cudaMemcpy2DAsync(d[k], dp, h[k], tile->pitch, dp, tile->n_sites, cudaMemcpyHostToDevice, s.stream));
        }
        if (tile->n_sites)
            BV_CUDA(ctx, cudaMemcpyAsync(s.d_ref, tile->ref_base, tile->n_sites, cudaMemcpyHostToDevice, s.stream));
        s.qual_host = qual_zero_copy;
        s.h2d_bytes = (size_t)tile->n_sites * dp * (qual_zero_copy ? 2 : 3) + tile->n_sites;
        dev.base = d[0]; dev.qual = d[1]; dev.strand = d[2]; dev.ref_base = s.d_ref;
        dev.pitch = dp;
        dev.location = BV_LOC_DEVICE;
    }
    int rc = fill_kernel_args(ctx, &dev, s.d_out, s.scratch, a);
    if (rc != BV_OK) return rc;
    if (s.qual_host) { a->qual = s.qual_host; a->qual_pitch = tile->pitch; }
    if (!with_calls) return BV_OK;
    bv_tile_aux dev_aux = *aux;
    bool aux_in_place = false;
    if (tile->location == BV_LOC_HOST && tile->n_sites) {
        // the aux planes are read for the called rows only: in place when pinned, else uploaded whole
        const uint8_t* zm = static_cast<const uint8_t*>(host_device_pointer(aux->mapq));
        const uint16_t* zr = static_cast<const uint16_t*>(host_device_pointer(aux->rpr));
        if (aux->rpr_pitch % 8 != 0 || aux->rpr_pitch < tile->n_samples) return set_err(ctx, BV_ERR_ARG, "bv_tile_aux: bad rpr_pitch");
        aux_in_place = zm && zr;
        if (aux_in_place) {
            dev_aux.mapq = zm; dev_aux.rpr = zr;
        } else {
            const size_t plane = (size_t)ctx->prm.max_sites * ctx->pitch_cap;
            if (!s.d_aux) BV_CUDA(ctx, cudaMalloc(&s.d_aux, 3 * plane));
            const uint64_t dp = dev.pitch;
            BV_CUDA(ctx, cudaMemcpy2DAsync(s.d_aux, dp, aux->mapq, tile->pitch, dp, tile->n_sites, cudaMemcpyHostToDevice, s.stream));
            BV_CUDA(ctx, cudaMemcpy2DAsync(s.d_aux + plane, 2 * dp, aux->rpr, 2 * aux->rpr_pitch, 2 * (size_t)tile->n_samples, tile->n_sites,
                                           cudaMemcpyHostToDevice, s.stream));
            s.h2d_bytes += (size_t)tile->n_sites * (dp + 2 * (size_t)tile->n_samples);
            dev_aux.mapq = s.d_aux; dev_aux.rpr = reinterpret_cast<const uint16_t*>(s.d_aux + plane); dev_aux.rpr_pitch = dp;
        }
    }
    rc = set_call_args(ctx, &dev, &dev_aux, s.scratch, s.h_calls, s.h_groups, a);
    if (aux_in_place) a->aux_pitch = tile->pitch;   // (the caller's planes keep the caller's pitch)
    return rc;
}

// Sparse host tile: upload the covered cells (4 or 2 bytes each) and expand them into the slot's dense planes (K0).  The qual
// plane -- and for the called-site kernels the mapq / rpr planes -- are device resident here (there is no host plane to read in
// place).  Fills `a` and s.h2d_bytes; trace: records the first two events of the tile's timeline.
static int upload_sparse(bv_ctx* ctx, bv_slot& s, const bv_sparse_tile* t, bool with_calls, bool trace, bv::SiteKernelArgs* a) {
    const bool u16 = t->format == BV_CELLS_U16;
    const size_t word_bytes = u16 ? sizeof(uint16_t) : sizeof(uint32_t);
    const uint64_t n_cells = t->n_sites ? t->site_start[t->n_sites] : 0;   // words of `format`
    if (n_cells > s.cells_cap) {   // grows only; sized by the first tiles of a run
        if (s.d_cells) BV_CUDA(ctx, cudaFree(s.d_cells));
        s.d_cells = nullptr; s.cells_cap = 0;
        const uint64_t cap = n_cells + n_cells / 4 + 1024;
        BV_CUDA(ctx, cudaMalloc(&s.d_cells, 2 * cap * sizeof(uint32_t)));
        s.cells_cap = cap;
    }
    if (!s.d_site_start) BV_CUDA(ctx, cudaMalloc(&s.d_site_start, ((size_t)ctx->prm.max_sites + 1) * sizeof(uint32_t)));
    const uint64_t dp = ((uint64_t)t->n_samples + 15) / 16 * 16;
    const size_t plane = (size_t)ctx->prm.max_sites * ctx->pitch_cap;
    if (with_calls && !s.d_aux) BV_CUDA(ctx, cudaMalloc(&s.d_aux, 3 * plane));
    bv_tile dev;
    dev.base = s.d_planes; dev.qual = s.d_planes + plane; dev.strand = s.d_planes + 2 * plane; dev.ref_base = s.d_ref;
    dev.pitch = dp; dev.n_sites = t->n_sites; dev.n_samples = t->n_samples; dev.location = BV_LOC_DEVICE; dev.out_mode = BV_OUT_RECORDS;
    int rc = fill_kernel_args(ctx, &dev, s.d_out, s.scratch, a);
    if (rc != BV_OK) return rc;
    if (with_calls) {
        bv_tile_aux dev_aux;
        dev_aux.mapq = s.d_aux; dev_aux.rpr = reinterpret_cast<const uint16_t*>(s.d_aux + plane); dev_aux.rpr_pitch = dp;
        rc = set_call_args(ctx, &dev, &dev_aux, s.scratch, s.h_calls, s.h_groups, a);
        if (rc != BV_OK) return rc;
    }
    // Uploads go through ONE stream, in submit order.  On the slots' own streams the uploads of the tiles in flight run side by
    // side and share the link: they all finish together, then their kernels run with the link idle, and the pipeline moves in
    // waves (100,000-sample tiles, 4 slots: 75 % of the bare-copy rate; profiles/r02_tile_timeline.txt).  First in, first out,
    // tile k's kernels run under tile k + 1's upload.
    cudaStream_t up = ctx->copy_stream;
    if (trace) {
        if (!ctx->ev_trace0) {
            BV_CUDA(ctx, cudaEventCreate(&ctx->ev_trace0));
            BV_CUDA(ctx, cudaEventRecord(ctx->ev_trace0, up));
            ctx->t_trace0 = host_seconds();
        }
        for (int k = 0; k < 4; ++k) if (!s.ev_trace[k]) BV_CUDA(ctx, cudaEventCreate(&s.ev_trace[k]));
        s.tile_no = ctx->tiles_traced++;
        s.t_submit = host_seconds() - ctx->t_trace0;
        BV_CUDA(ctx, cudaEventRecord(s.ev_trace[0], up));
    }
    if (t->n_sites && t->n_samples) {
        // (the small arrays first: when they come from pageable memory the call waits for what is queued in front of them.  Sending
        // them down the slot's own stream instead, out of the queue, was measured slower: C2 4.25 -> 5.6 ms per step, gpurun r02c6)
        BV_CUDA(ctx, cudaMemcpyAsync(s.d_site_start, t->site_start, ((size_t)t->n_sites + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, up));
        BV_CUDA(ctx, cudaMemcpyAsync(s.d_ref, t->ref_base, t->n_sites, cudaMemcpyHostToDevice, up));
        if (n_cells) {
            BV_CUDA(ctx, cudaMemcpyAsync(s.d_cells, t->cells, n_cells * word_bytes, cudaMemcpyHostToDevice, up));
            if (with_calls)
                BV_CUDA(ctx, cudaMemcpyAsync(s.d_cells + s.cells_cap, t->cells_aux, n_cells * sizeof(uint32_t), cudaMemcpyHostToDevice, up));
        }
        s.h2d_bytes = n_cells * (word_bytes + (with_calls ? sizeof(uint32_t) : 0)) + ((size_t)t->n_sites + 1) * sizeof(uint32_t) + t->n_sites;
        if (trace) BV_CUDA(ctx, cudaEventRecord(s.ev_trace[1], up));
        BV_CUDA(ctx, cudaEventRecord(s.ev_up, up));
        BV_CUDA(ctx, cudaStreamWaitEvent(s.stream, s.ev_up, 0));
        BV_CUDA(ctx, cudaMemsetAsync(a->counters, 0, bv::kNumCounters * sizeof(uint32_t), s.stream));
        bv::ExpandArgs x;
        x.cells = s.d_cells; x.cells_aux = with_calls ? s.d_cells + s.cells_cap : nullptr; x.site_start = s.d_site_start;
        x.base = s.d_planes; x.qual = s.d_planes + plane; x.strand = s.d_planes + 2 * plane;
        x.mapq = with_calls ? s.d_aux : nullptr;
        x.rpr = with_calls ? reinterpret_cast<uint16_t*>(s.d_aux + plane) : nullptr;
        x.counters = a->counters;
        x.pitch = dp; x.rpr_pitch = dp; x.n_cells = n_cells; x.n_sites = t->n_sites; x.n_samples = t->n_samples;
        uint32_t grid = (t->n_sites + bv::kExpandWarps - 1) / bv::kExpandWarps;
        const uint32_t cap = (uint32_t)ctx->num_sms * 2u;   // persistent: 2 CTAs of 16 warps per SM (96 KB of staging each)
        if (grid > cap) grid = cap;
        if (u16) bv::bv_expand_kernel<BV_CELLS_U16><<<grid, bv::kExpandWarps * 32, bv::kExpandSmemBytes, s.stream>>>(x);
        else bv::bv_expand_kernel<BV_CELLS_U32><<<grid, bv::kExpandWarps * 32, bv::kExpandSmemBytes, s.stream>>>(x);
        BV_CUDA(ctx, cudaGetLastError());
        ctx->launches += 1;
    }
    return BV_OK;
}

// Everything after the upload of a slot's tile, on the slot's stream: K1..K6; with lists their upload, K8 (per site, or over the
// packed list of a compact tile) and its results back; the records back into dst; the counters back for the slots whose wait reads
// them (sparse, called-site or compact tiles); and the slot's bookkeeping.  trace: the last two events of a traced tile.
static int submit_tail(bv_ctx* ctx, bv_slot& s, bv::SiteKernelArgs& a, bool with_calls, bool with_lists, uint32_t n_listed,
                       bool counters_zeroed, bool trace, bv_site_out* dst) {
    const uint32_t n_sites = a.n_sites;
    if (s.compact) {
        a.brief = s.d_brief;
        a.full_out = static_cast<bv_site_out*>(const_cast<void*>(host_device_pointer(s.h_out)));
        if (!a.full_out) return set_err(ctx, BV_ERR_CUDA, "pinned staging is not device accessible");
    }
    int rc = launch_site_kernel(ctx, a, s.stream, counters_zeroed);
    if (rc != BV_OK) return rc;
    const bool packed = with_lists && s.compact;
    const uint32_t n_lrt = packed ? n_listed : n_sites;
    if (with_lists && n_lrt) {
        const size_t list_bytes = (size_t)n_lrt * (packed ? sizeof(uint2) : sizeof(uint32_t));
        BV_CUDA(ctx, cudaMemcpyAsync(s.d_lists, s.h_lists, list_bytes, cudaMemcpyHostToDevice, s.stream));
        rc = launch_list_kernel(ctx, a, s.d_lists, packed ? reinterpret_cast<const uint2*>(s.d_lists) : nullptr, n_lrt, s.d_lrt, s.stream);
        if (rc != BV_OK) return rc;
        BV_CUDA(ctx, cudaMemcpyAsync(s.h_lrt, s.d_lrt, (size_t)n_lrt * sizeof(bv_lrt_out), cudaMemcpyDeviceToHost, s.stream));
        s.h2d_bytes += list_bytes;
    }
    if (trace) BV_CUDA(ctx, cudaEventRecord(s.ev_trace[2], s.stream));
    rc = return_records(ctx, s, a, n_sites, dst);
    if (rc != BV_OK) return rc;
    if (s.sparse || with_calls || s.compact) {   // (a tile without cells leaves them zero)
        memset(s.h_counters, 0, bv::kNumCounters * sizeof(uint32_t));
        if (n_sites && a.n_samples)
            BV_CUDA(ctx, cudaMemcpyAsync(s.h_counters, a.counters, bv::kNumCounters * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
    }
    if (trace) BV_CUDA(ctx, cudaEventRecord(s.ev_trace[3], s.stream));
    s.with_calls = with_calls;
    s.with_lists = with_lists;
    s.lists_packed = packed;
    s.n_listed = n_listed;
    s.n_sites = n_sites;
    s.busy = true;
    ctx->h2d_bytes_total += s.h2d_bytes;
    return BV_OK;
}

// Dense tile, host or device resident (bv_tile_submit, _calls, _lists).
static int tile_submit_dense(bv_ctx* ctx, int slot, const bv_tile* tile, const bv_tile_aux* aux, bool with_calls,
                             const uint8_t (*lists)[4] = nullptr) {
    BvRange range("bv_tile_submit (dense tile: H2D, kernels, D2H)");
    bv_slot* sp = slot_of(ctx, slot);
    if (!sp) return BV_ERR_ARG;
    if (!tile) return set_err(ctx, BV_ERR_ARG, "null tile");
    bv_slot& s = *sp;
    if (s.busy) return set_err(ctx, BV_ERR_STATE, "slot %d is busy: call bv_tile_wait first", slot);
    if (tile->n_sites > ctx->prm.max_sites) return set_err(ctx, BV_ERR_ARG, "tile has %u sites > max_sites %u", tile->n_sites, ctx->prm.max_sites);
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    s.qual_host = nullptr;
    s.h2d_bytes = 0;
    s.sparse = false; s.out_direct = false; s.out_user = nullptr;
    s.compact = tile->location == BV_LOC_HOST && tile->out_mode == BV_OUT_COMPACT;
    s.h_ref = tile->location == BV_LOC_HOST ? tile->ref_base : nullptr;
    if (with_calls && tile->location == BV_LOC_DEVICE && tile->out_mode == BV_OUT_COMPACT)
        return set_err(ctx, BV_ERR_ARG, "BV_OUT_COMPACT: device-resident tiles have no compact form");
    uint32_t n_listed = 0;
    if (lists) {
        if (tile->out_mode != BV_OUT_RECORDS) return set_err(ctx, BV_ERR_ARG, "bv_tile_submit_lists: out_mode must be BV_OUT_RECORDS");
        const int rc = stage_lists(ctx, s, lists, tile->n_sites, false, &n_listed);
        if (rc != BV_OK) return rc;
    }
    bv::SiteKernelArgs a;
    int rc = upload_dense(ctx, s, tile, aux, with_calls, &a);
    if (rc != BV_OK) return rc;
    return submit_tail(ctx, s, a, with_calls, lists != nullptr, n_listed, false, false, s.h_out);
}

// Sparse host tile (bv_tile_submit_sparse, _calls, _lists): the cells up, K0 expand, then what a dense tile runs.
static int tile_submit_sparse(bv_ctx* ctx, int slot, const bv_sparse_tile* t, bool with_calls, const uint8_t (*lists)[4] = nullptr) {
    BvRange range("bv_tile_submit_sparse (H2D of the cells, K0 expand, kernels, D2H)");
    bv_slot* sp = slot_of(ctx, slot);
    if (!sp) return BV_ERR_ARG;
    if (!t) return set_err(ctx, BV_ERR_ARG, "null tile");
    bv_slot& s = *sp;
    if (s.busy) return set_err(ctx, BV_ERR_STATE, "slot %d is busy: call bv_tile_wait first", slot);
    if (t->n_sites > ctx->prm.max_sites) return set_err(ctx, BV_ERR_ARG, "tile has %u sites > max_sites %u", t->n_sites, ctx->prm.max_sites);
    if (t->n_samples > ctx->prm.max_samples || t->n_samples > BV_CELL_MAX_SAMPLES)
        return set_err(ctx, BV_ERR_ARG, "sparse tile: n_samples %u > max_samples %u or > %u", t->n_samples, ctx->prm.max_samples, BV_CELL_MAX_SAMPLES);
    if (t->n_sites && (!t->site_start || !t->ref_base)) return set_err(ctx, BV_ERR_ARG, "bv_sparse_tile: null pointer");
    if (t->format != BV_CELLS_U32 && t->format != BV_CELLS_U16) return set_err(ctx, BV_ERR_ARG, "bv_sparse_tile: unknown format %u", t->format);
    const bool u16 = t->format == BV_CELLS_U16;
    const uint64_t n_cells = t->n_sites ? t->site_start[t->n_sites] : 0;   // words of `format`
    if (t->n_sites && t->site_start[0] != 0) return set_err(ctx, BV_ERR_ARG, "bv_sparse_tile: site_start[0] must be 0");
    if (n_cells && (!t->cells || (with_calls && !t->cells_aux))) return set_err(ctx, BV_ERR_ARG, "bv_sparse_tile: null cells");
    if (n_cells > (uint64_t)t->n_sites * ((uint64_t)t->n_samples + (u16 ? t->n_samples / BV_CELL16_GAP_SKIP + 2u : 0u)))
        return set_err(ctx, BV_ERR_ARG, "bv_sparse_tile: more cells than sample-sites");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    s.qual_host = nullptr;
    s.h2d_bytes = 0;
    s.sparse = true; s.out_direct = false; s.out_user = t->out;
    s.compact = t->out_mode == BV_OUT_COMPACT;
    s.h_ref = t->ref_base;
    if (s.compact && t->out) return set_err(ctx, BV_ERR_ARG, "BV_OUT_COMPACT: `out` must be NULL");
    uint32_t n_listed = 0;
    if (lists) {
        const int rc = stage_lists(ctx, s, lists, t->n_sites, s.compact, &n_listed);
        if (rc != BV_OK) return rc;
    }
    const bool trace = ctx->trace && t->n_sites && t->n_samples;
    bv::SiteKernelArgs a;
    int rc = upload_sparse(ctx, s, t, with_calls, trace, &a);
    if (rc != BV_OK) return rc;
    // pinned records of the caller: the D2H copy goes straight into them
    s.out_direct = t->n_sites && t->out && host_device_pointer(t->out);
    return submit_tail(ctx, s, a, with_calls, lists != nullptr, n_listed, true, trace, s.out_direct ? t->out : s.h_out);
}

int bv_tile_submit(bv_ctx* ctx, int slot, const bv_tile* tile) { return tile_submit_dense(ctx, slot, tile, nullptr, false); }

int bv_tile_submit_calls(bv_ctx* ctx, int slot, const bv_tile* tile, const bv_tile_aux* aux) {
    if (!aux) return set_err(ctx, BV_ERR_ARG, "bv_tile_submit_calls: null aux");
    return tile_submit_dense(ctx, slot, tile, aux, true);
}

int bv_tile_submit_lists(bv_ctx* ctx, int slot, const bv_tile* tile, const uint8_t (*lists)[4]) {
    if (!lists) return set_err(ctx, BV_ERR_ARG, "bv_tile_submit_lists: null lists");
    return tile_submit_dense(ctx, slot, tile, nullptr, false, lists);
}

int bv_tile_submit_sparse(bv_ctx* ctx, int slot, const bv_sparse_tile* tile) { return tile_submit_sparse(ctx, slot, tile, false); }
int bv_tile_submit_sparse_calls(bv_ctx* ctx, int slot, const bv_sparse_tile* tile) { return tile_submit_sparse(ctx, slot, tile, true); }
int bv_tile_submit_sparse_lists(bv_ctx* ctx, int slot, const bv_sparse_tile* tile, const uint8_t (*lists)[4]) {
    if (tile && tile->n_sites && !lists) return set_err(ctx, BV_ERR_ARG, "bv_tile_submit_sparse_lists: null lists");
    static const uint8_t no_lists[1][4] = {{BV_LIST_END, BV_LIST_END, BV_LIST_END, BV_LIST_END}};   // (an empty tile may pass NULL)
    return tile_submit_sparse(ctx, slot, tile, false, lists ? lists : no_lists);
}

uint64_t bv_sparse_encode16_bound(uint64_t n_cells, uint32_t n_sites, uint32_t n_samples) {
    return n_cells + (uint64_t)n_sites * (n_samples / BV_CELL16_GAP_SKIP + 1u);   // at most n_samples / 31 skips per site
}

int bv_sparse_encode16(const uint32_t* cells, const uint32_t* aux32, const uint32_t* site_start, uint32_t n_sites,
                       uint16_t* words16, uint32_t* aux16, uint64_t max_words, uint32_t* start16, uint64_t* n_words) {
    if (!site_start || !n_words || (n_sites && site_start[n_sites] && !cells)) return set_err(nullptr, BV_ERR_ARG, "null argument");
    uint64_t n = 0;
    static const bool have_avx2 = bv::encode16_have_avx2() && !getenv("BASEVAR_B200_NO_AVX2");
    for (uint32_t s = 0; s < n_sites; ++s) {
        if (start16) start16[s] = (uint32_t)n;
        const uint32_t c0 = site_start[s], c1 = site_start[s + 1];
        if (c1 < c0) return set_err(nullptr, BV_ERR_ARG, "site_start does not ascend at site %u", s);
        uint32_t next = 0;   // the sample index a gap of 0 would mean
        // room for the worst case of this site: every cell plus a skip word per 31 samples of the 2^20 a cell can name
        const bool roomy = words16 && n + (uint64_t)(c1 - c0) + BV_CELL_MAX_SAMPLES / BV_CELL16_GAP_SKIP + 1 <= max_words;
        // the vector loop stores eight words at a time, so it wants eight words of slack behind the worst case
        const bool wide = roomy && c1 - c0 >= 16 && n + (uint64_t)(c1 - c0) + BV_CELL_MAX_SAMPLES / BV_CELL16_GAP_SKIP + 9 <= max_words && have_avx2;
        for (uint32_t c = c0; c < c1; ++c) {
            if (roomy) {
                uint16_t* o = words16 + n;
                uint32_t* oa = aux16 ? aux16 + n : nullptr;
                const uint32_t* stop =
                    wide ? (aux16 ? bv::encode16_run_avx2<true>(cells + c, cells + c1, aux32 ? aux32 + c1 : nullptr, o, oa, next)
                                  : bv::encode16_run_avx2<false>(cells + c, cells + c1, nullptr, o, oa, next))
                         : (aux16 ? encode16_run<true>(cells + c, cells + c1, aux32 ? aux32 + c1 : nullptr, o, oa, next)
                                  : encode16_run<false>(cells + c, cells + c1, nullptr, o, oa, next));
                n = (uint64_t)(o - words16);
                c = (uint32_t)(stop - cells);
                if (c >= c1) break;
            }
            const uint32_t w = cells[c], i = w & (BV_CELL_MAX_SAMPLES - 1u), strand = (w >> 23) & 3u;
            if (i < next) return set_err(nullptr, BV_ERR_ARG, "site %u: cells do not ascend by sample (BV_CELLS_U16 needs them to)", s);
            if (strand > BV_STRAND_REV) return set_err(nullptr, BV_ERR_ARG, "site %u, sample %u: strand code %u has no 16-bit form", s, i, strand);
            uint32_t g = i - next;
            while (g >= BV_CELL16_GAP_SKIP) {
                if (words16) {
                    if (n >= max_words) return set_err(nullptr, BV_ERR_ARG, "more than max_words words");
                    words16[n] = (uint16_t)BV_CELL16_GAP_SKIP;
                    if (aux16) aux16[n] = 0;
                }
                ++n;
                g -= BV_CELL16_GAP_SKIP;
            }
            if (words16) {
                if (n >= max_words) return set_err(nullptr, BV_ERR_ARG, "more than max_words words");
                words16[n] = BV_CELL16_PACK(g, (w >> 20) & 7u, strand, w >> 25);
                if (aux16) aux16[n] = aux32 ? aux32[c] : 0;
            }
            ++n;
            next = i + 1;
        }
        if (n > 0xffffffffull) return set_err(nullptr, BV_ERR_ARG, "more than 2^32 words in one tile");
    }
    if (start16) start16[n_sites] = (uint32_t)n;
    *n_words = n;
    return BV_OK;
}

int bv_synth_fill_sparse_host(const bv_synth_model* model, uint64_t site0, uint32_t n_sites, uint32_t n_samples,
                              uint32_t* cells, uint32_t* cells_aux, uint64_t max_cells, uint32_t* site_start,
                              uint8_t* ref_base, uint64_t* n_cells) {
    if (!model || !n_cells) return set_err(nullptr, BV_ERR_ARG, "null argument");
    if (n_samples > BV_CELL_MAX_SAMPLES) return set_err(nullptr, BV_ERR_ARG, "n_samples > %u", BV_CELL_MAX_SAMPLES);
    uint64_t n = 0;
    for (uint32_t s = 0; s < n_sites; ++s) {
        const bv::SynthSite ss = bv::synth_site(model, site0 + s);
        if (ref_base) ref_base[s] = "ACGT"[ss.ref];
        if (site_start) site_start[s] = (uint32_t)n;
        for (uint32_t i = 0; i < n_samples; ++i) {
            const bv::SynthCell c = bv::synth_cell(model, ss, i);
            if (c.base == BV_BASE_N) continue;   // the generator makes N only for uncovered cells
            if (cells) {
                if (n >= max_cells) return set_err(nullptr, BV_ERR_ARG, "more than max_cells cells");
                cells[n] = BV_CELL_PACK(i, c.base, c.strand, c.qual);
                if (cells_aux) cells_aux[n] = BV_CELL_AUX_PACK(c.mapq, bv::synth_rpr(model, ss, i));
            }
            ++n;
        }
        if (n > 0xffffffffull) return set_err(nullptr, BV_ERR_ARG, "more than 2^32 cells in one tile");
    }
    if (site_start) site_start[n_sites] = (uint32_t)n;
    *n_cells = n;
    return BV_OK;
}

// The wait of every form: synchronise the slot, print its trace line, report bad cells; then the records into `out` (and into the
// sparse tile's `out`), or with `brief` the views of a compact tile's pinned staging.
static int wait_slot(bv_ctx* ctx, int slot, bv_slot& s, bv_site_out* out, const bv_site_brief** brief = nullptr,
                     const bv_site_out** full = nullptr, uint32_t* n_full = nullptr) {
    BvRange range("bv_tile_wait");
    if (!s.busy) return set_err(ctx, BV_ERR_STATE, "slot %d has nothing submitted", slot);
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    const double t_wait0 = ctx->trace ? host_seconds() - ctx->t_trace0 : 0.0;
    cudaError_t e = cudaStreamSynchronize(s.stream);
    s.busy = false;
    BV_CUDA(ctx, e);
    if (ctx->trace && s.sparse && s.ev_trace[3] && s.n_sites) {
        float ms[4] = {0, 0, 0, 0};
        for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&ms[k], ctx->ev_trace0, s.ev_trace[k]);
        fprintf(stderr, "bv trace: tile %llu slot %d: submit at %.3f ms (host); upload %.3f .. %.3f, kernels until %.3f, results back %.3f (device); "
                        "wait %.3f .. %.3f (host); %.1f MB up\n",
                (unsigned long long)s.tile_no, slot, 1e3 * s.t_submit, ms[0], ms[1], ms[2], ms[3], 1e3 * t_wait0,
                1e3 * (host_seconds() - ctx->t_trace0), s.h2d_bytes / 1e6);
    }
    if (s.sparse && s.n_sites && s.h_counters[bv::kCntBadCell])
        return set_err(ctx, BV_ERR_ARG, "sparse tile: cell with sample >= n_samples or site_start not ascending / beyond the cell count");
    if (s.compact) {   // collected in compact form (bv_tile_wait_compact), or expanded here for a caller that wants records
        if (brief) {
            *brief = s.h_brief; *full = s.h_out; *n_full = s.n_sites ? s.h_counters[bv::kCntFull] : 0;
        } else if (out) {
            const uint32_t n_full = s.h_counters[bv::kCntFull];
            for (uint32_t i = 0; i < s.n_sites; ++i) {
                const bv_site_brief& b = s.h_brief[i];
                if (b.w0 & 0x80000000u) {
                    const uint32_t k = b.w0 & 0x7fffffffu;
                    if (k >= n_full) return set_err(ctx, BV_ERR_STATE, "compact tile: record index out of range");
                    out[i] = s.h_out[k];
                } else bv_site_expand(&b, s.h_ref ? s.h_ref[i] : 0, ctx->prm.min_af, &out[i]);
            }
        }
        return BV_OK;
    }
    const bv_site_out* rec = s.out_direct ? s.out_user : s.h_out;
    if (s.out_user && !s.out_direct && s.n_sites) memcpy(s.out_user, s.h_out, (size_t)s.n_sites * sizeof(bv_site_out));
    if (out && out != rec && s.n_sites) memcpy(out, rec, (size_t)s.n_sites * sizeof(bv_site_out));
    return BV_OK;
}

int bv_tile_wait(bv_ctx* ctx, int slot, bv_site_out* out) {
    bv_slot* s = slot_of(ctx, slot);
    return s ? wait_slot(ctx, slot, *s, out) : BV_ERR_ARG;
}

int bv_tile_wait_compact(bv_ctx* ctx, int slot, const bv_site_brief** brief, const bv_site_out** full, uint32_t* n_full) {
    bv_slot* s = slot_of(ctx, slot);
    if (!s) return BV_ERR_ARG;
    if (!brief || !full || !n_full) return set_err(ctx, BV_ERR_ARG, "bv_tile_wait_compact: null argument");
    if (s->busy && !s->compact) return set_err(ctx, BV_ERR_STATE, "slot %d was not submitted with BV_OUT_COMPACT", slot);
    return wait_slot(ctx, slot, *s, nullptr, brief, full, n_full);
}

void bv_site_expand(const bv_site_brief* b, uint8_t ref_base, float min_af, bv_site_out* out) {
    memset(out, 0, sizeof(*out));
    if (!b || (b->w0 & 0x80000000u) || b->w0 == 0) return;
    unsigned rc = ref_base;
    if (rc >= 'a' && rc <= 'z') rc -= 32;
    const int code = rc == 'A' ? 0 : rc == 'C' ? 1 : rc == 'G' ? 2 : rc == 'T' ? 3 : -1;
    if (code < 0) return;
    out->depth[code] = b->w0;
    out->fwd[code] = b->w0 - b->w1;
    out->rev[code] = b->w1;
    // one active allele (the reference's single-column EM: f = 1, no ALT) when 1.0 >= min_af
    const uint8_t n_active = (1.0 >= (double)min_af) ? 1 : 0;
    out->n_active = n_active;
    out->em_calls = n_active;
}

// The called-site outputs of a waited-for slot into the caller's arrays.
static int copy_calls(bv_ctx* ctx, const bv_slot& s, bv_call_out* calls, uint32_t max_calls, uint32_t* n_calls, bv_group_out* groups) {
    const uint32_t n = s.h_counters[bv::kCntCalled];
    *n_calls = n;
    if (n > max_calls) return set_err(ctx, BV_ERR_ARG, "tile has %u called sites > max_calls %u", n, max_calls);
    if (n && calls) memcpy(calls, s.h_calls, (size_t)n * sizeof(bv_call_out));
    if (n && groups && ctx->n_groups && s.h_groups) memcpy(groups, s.h_groups, (size_t)n * ctx->n_groups * sizeof(bv_group_out));
    return BV_OK;
}

int bv_tile_wait_calls(bv_ctx* ctx, int slot, bv_site_out* out, bv_call_out* calls, uint32_t max_calls,
                       uint32_t* n_calls, bv_group_out* groups) {
    bv_slot* s = slot_of(ctx, slot);
    if (!s) return BV_ERR_ARG;
    if (!n_calls) return set_err(ctx, BV_ERR_ARG, "bv_tile_wait_calls: null n_calls");
    if (s->busy && !s->with_calls) return set_err(ctx, BV_ERR_STATE, "slot %d was submitted without called-site kernels", slot);
    int rc = wait_slot(ctx, slot, *s, out);
    if (rc != BV_OK) return rc;
    return copy_calls(ctx, *s, calls, max_calls, n_calls, groups);
}

int bv_tile_wait_calls_compact(bv_ctx* ctx, int slot, const bv_site_brief** brief, const bv_site_out** full, uint32_t* n_full,
                               bv_call_out* calls, uint32_t max_calls, uint32_t* n_calls, bv_group_out* groups) {
    bv_slot* s = slot_of(ctx, slot);
    if (!s) return BV_ERR_ARG;
    if (!n_calls) return set_err(ctx, BV_ERR_ARG, "bv_tile_wait_calls_compact: null n_calls");
    if (s->busy && !s->with_calls) return set_err(ctx, BV_ERR_STATE, "slot %d was submitted without called-site kernels", slot);
    int rc = bv_tile_wait_compact(ctx, slot, brief, full, n_full);
    if (rc != BV_OK) return rc;
    return copy_calls(ctx, *s, calls, max_calls, n_calls, groups);
}

int bv_tile_wait_lists(bv_ctx* ctx, int slot, bv_site_out* out, bv_lrt_out* lrt_out) {
    bv_slot* s = slot_of(ctx, slot);
    if (!s) return BV_ERR_ARG;
    if (!lrt_out) return set_err(ctx, BV_ERR_ARG, "bv_tile_wait_lists: null lrt_out");
    if (s->busy && !s->with_lists) return set_err(ctx, BV_ERR_STATE, "slot %d was submitted without lists", slot);
    if (s->busy && s->lists_packed) return set_err(ctx, BV_ERR_STATE, "slot %d has compact results: collect with bv_tile_wait_lists_compact", slot);
    int rc = wait_slot(ctx, slot, *s, out);
    if (rc != BV_OK) return rc;
    if (s->n_sites) memcpy(lrt_out, s->h_lrt, (size_t)s->n_sites * sizeof(bv_lrt_out));
    return BV_OK;
}

int bv_tile_wait_lists_compact(bv_ctx* ctx, int slot, const bv_site_brief** brief, const bv_site_out** full, uint32_t* n_full,
                               bv_lrt_out* lrt_out, uint32_t max_lrt, uint32_t* n_lrt) {
    bv_slot* s = slot_of(ctx, slot);
    if (!s) return BV_ERR_ARG;
    if (!n_lrt) return set_err(ctx, BV_ERR_ARG, "bv_tile_wait_lists_compact: null n_lrt");
    if (s->busy && !s->lists_packed) return set_err(ctx, BV_ERR_STATE, "slot %d was not submitted with lists and BV_OUT_COMPACT", slot);
    int rc = bv_tile_wait_compact(ctx, slot, brief, full, n_full);
    if (rc != BV_OK) return rc;
    const uint32_t n = s->n_listed;
    *n_lrt = n;
    if (n > max_lrt) return set_err(ctx, BV_ERR_ARG, "tile has %u listed sites > max_lrt %u", n, max_lrt);
    if (n && !lrt_out) return set_err(ctx, BV_ERR_ARG, "bv_tile_wait_lists_compact: null lrt_out");
    if (n) memcpy(lrt_out, s->h_lrt, (size_t)n * sizeof(bv_lrt_out));
    return BV_OK;
}

int bv_synth_fill_rpr_device(bv_ctx* ctx, uint64_t site0, uint32_t n_sites, uint32_t n_samples, uint64_t rpr_pitch,
                             uint16_t* d_rpr, void* stream) {
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    if (!ctx->has_model) return set_err(ctx, BV_ERR_STATE, "bv_synth_set_model was not called");
    if (!d_rpr || rpr_pitch % 8 != 0 || rpr_pitch < n_samples) return set_err(ctx, BV_ERR_ARG, "bad rpr plane / pitch");
    if (n_sites == 0) return BV_OK;
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t units = (uint64_t)n_sites * (rpr_pitch >> 3);
    uint64_t blocks = (units + 255) / 256;
    const uint64_t cap = (uint64_t)ctx->num_sms * 32;
    if (blocks > cap) blocks = cap;
    bv::bv_synth_rpr_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(ctx->d_model, site0, n_sites, n_samples, rpr_pitch, d_rpr);
    BV_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BV_OK;
}

int bv_synth_fill_rpr_host(const bv_synth_model* model, uint64_t site0, uint32_t n_sites, uint32_t n_samples,
                           uint64_t rpr_pitch, uint16_t* rpr) {
    if (!model || !rpr || rpr_pitch < n_samples) return set_err(nullptr, BV_ERR_ARG, "bad argument");
    for (uint32_t s = 0; s < n_sites; ++s) {
        const bv::SynthSite ss = bv::synth_site(model, site0 + s);
        for (uint64_t i = 0; i < rpr_pitch; ++i) rpr[(size_t)s * rpr_pitch + i] = i < n_samples ? bv::synth_rpr(model, ss, i) : 0;
    }
    return BV_OK;
}

int bv_synth_set_model(bv_ctx* ctx, const bv_synth_model* model) {
    if (!ctx || !model) return set_err(ctx, BV_ERR_ARG, "bv_synth_set_model: null argument");
    if (model->q_lo + model->q_span > BV_QUAL_MAX + 1) return set_err(ctx, BV_ERR_ARG, "synthetic phred range exceeds 93");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->d_model) BV_CUDA(ctx, cudaMalloc(&ctx->d_model, sizeof(bv_synth_model)));
    BV_CUDA(ctx, cudaMemcpy(ctx->d_model, model, sizeof(bv_synth_model), cudaMemcpyHostToDevice));
    ctx->has_model = true;
    return BV_OK;
}

int bv_synth_fill_device(bv_ctx* ctx, uint64_t site0, uint32_t n_sites, uint32_t n_samples, uint64_t pitch,
                         uint8_t* d_base, uint8_t* d_qual, uint8_t* d_strand, uint8_t* d_mapq, uint8_t* d_ref_base,
                         void* stream) {
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    if (!ctx->has_model) return set_err(ctx, BV_ERR_STATE, "bv_synth_set_model was not called");
    if (!d_base || !d_qual || !d_strand || !d_ref_base) return set_err(ctx, BV_ERR_ARG, "null plane");
    if (pitch % 16 != 0 || pitch < n_samples) return set_err(ctx, BV_ERR_ARG, "bad pitch");
    if (n_sites == 0) return BV_OK;
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t units = (uint64_t)n_sites * (pitch >> 4);
    uint64_t blocks = (units + 255) / 256;
    const uint64_t cap = (uint64_t)ctx->num_sms * 32;
    if (blocks > cap) blocks = cap;
    bv::bv_synth_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(ctx->d_model, site0, n_sites, n_samples, pitch,
                                                                        d_base, d_qual, d_strand, d_mapq, d_ref_base);
    BV_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return BV_OK;
}

int bv_synth_fill_host(const bv_synth_model* model, uint64_t site0, uint32_t n_sites, uint32_t n_samples, uint64_t pitch,
                       uint8_t* base, uint8_t* qual, uint8_t* strand, uint8_t* mapq, uint8_t* ref_base) {
    if (!model || !base || !qual || !strand || !ref_base) return set_err(nullptr, BV_ERR_ARG, "null argument");
    if (pitch < n_samples) return set_err(nullptr, BV_ERR_ARG, "bad pitch");
    for (uint32_t s = 0; s < n_sites; ++s) {
        const bv::SynthSite ss = bv::synth_site(model, site0 + s);
        ref_base[s] = "ACGT"[ss.ref];
        const size_t row = (size_t)s * pitch;
        for (uint64_t i = 0; i < pitch; ++i) {
            bv::SynthCell c;
            if (i < n_samples) c = bv::synth_cell(model, ss, i);
            else { c.base = BV_BASE_N; c.qual = 0; c.strand = BV_STRAND_NONE; c.mapq = 0; }
            base[row + i] = c.base; qual[row + i] = c.qual; strand[row + i] = c.strand;
            if (mapq) mapq[row + i] = c.mapq;
        }
    }
    return BV_OK;
}

int bv_fisher_fs(bv_ctx* ctx, const int32_t* tables, uint32_t n, double* fs_out) {
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    if (n == 0) return BV_OK;
    if (!tables || !fs_out) return set_err(ctx, BV_ERR_ARG, "bv_fisher_fs: null argument");
    for (uint32_t i = 0; i < n; ++i) {
        int64_t tot = 0;
        for (int k = 0; k < 4; ++k) {
            if (tables[4 * (size_t)i + k] < 0) return set_err(ctx, BV_ERR_ARG, "bv_fisher_fs: negative count in table %u", i);
            tot += tables[4 * (size_t)i + k];
        }
        // the log-factorial table holds lgamma(k + 1) for k <= max_samples + 1
        if (tot > (int64_t)ctx->prm.max_samples + 1) return set_err(ctx, BV_ERR_ARG, "bv_fisher_fs: table %u has %lld reads > max_samples + 1", i, (long long)tot);
    }
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    int4* d_t = nullptr;
    double* d_fs = nullptr;
    cudaError_t e = cudaMalloc(&d_t, (size_t)n * sizeof(int4));
    if (e == cudaSuccess) e = cudaMalloc(&d_fs, (size_t)n * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(d_t, tables, (size_t)n * sizeof(int4), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        bv::bv_fs_kernel<<<(n + 127) / 128, 128>>>(d_t, d_fs, n, ctx->d_logfact);
        e = cudaGetLastError();
        ctx->launches += 1;
    }
    if (e == cudaSuccess) e = cudaMemcpy(fs_out, d_fs, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost);
    cudaFree(d_t); cudaFree(d_fs);
    BV_CUDA(ctx, e);
    return BV_OK;
}

int bv_ranksum_test(bv_ctx* ctx, const uint8_t* bases, const int32_t* values, const uint64_t* start, const uint8_t* ref_base,
                    const uint8_t* alt_mask, uint32_t n, double* phred_out) {
    BvRange range("bv_ranksum_test (H2D, K9, D2H)");
    if (!ctx) return set_err(nullptr, BV_ERR_ARG, "null context");
    if (n == 0) return BV_OK;
    if (!start || !ref_base || !alt_mask || !phred_out) return set_err(ctx, BV_ERR_ARG, "bv_ranksum_test: null argument");
    if (start[0] != 0) return set_err(ctx, BV_ERR_ARG, "bv_ranksum_test: start[0] = %llu, not 0", (unsigned long long)start[0]);
    for (uint32_t p = 0; p < n; ++p) {
        if (start[p + 1] < start[p]) return set_err(ctx, BV_ERR_ARG, "bv_ranksum_test: start[%u] < start[%u]", p + 1, p);
        if (start[p + 1] - start[p] > ctx->prm.max_samples)
            return set_err(ctx, BV_ERR_ARG, "bv_ranksum_test: problem %u has %llu entries > max_samples %u", p,
                           (unsigned long long)(start[p + 1] - start[p]), ctx->prm.max_samples);
        if (alt_mask[p] > 15) return set_err(ctx, BV_ERR_ARG, "bv_ranksum_test: alt_mask[%u] = %u > 15", p, alt_mask[p]);
    }
    const uint64_t total = start[n];
    if (total && (!bases || !values)) return set_err(ctx, BV_ERR_ARG, "bv_ranksum_test: null bases / values");
    BV_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->rs_stream) {   // on first use: a context that never calls this sets up exactly what it did without it
        BV_CUDA(ctx, cudaFuncSetAttribute(bv::bv_ranksum_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bv::kRsSmemBytes));
        BV_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->rs_stream, cudaStreamNonBlocking));
    }
    if (total > ctx->rs_entries_cap) {   // (a failed allocation leaves the scratch empty, so the next call allocates again)
        cudaFree(ctx->d_rs_bases); cudaFree(ctx->d_rs_values);
        ctx->d_rs_bases = nullptr; ctx->d_rs_values = nullptr; ctx->rs_entries_cap = 0;
        BV_CUDA(ctx, cudaMalloc(&ctx->d_rs_bases, total));
        BV_CUDA(ctx, cudaMalloc(&ctx->d_rs_values, total * sizeof(int32_t)));
        ctx->rs_entries_cap = total;
    }
    if (n > ctx->rs_problems_cap) {
        cudaFree(ctx->d_rs_start); cudaFree(ctx->d_rs_ref); cudaFree(ctx->d_rs_out);
        ctx->d_rs_start = nullptr; ctx->d_rs_ref = nullptr; ctx->d_rs_out = nullptr; ctx->rs_problems_cap = 0;
        BV_CUDA(ctx, cudaMalloc(&ctx->d_rs_start, ((size_t)n + 1) * sizeof(uint64_t)));
        BV_CUDA(ctx, cudaMalloc(&ctx->d_rs_ref, 2 * (size_t)n));
        BV_CUDA(ctx, cudaMalloc(&ctx->d_rs_out, (size_t)n * sizeof(double)));
        ctx->rs_problems_cap = n;
    }
    cudaStream_t st = ctx->rs_stream;
    uint8_t* d_mask = ctx->d_rs_ref + ctx->rs_problems_cap;
    if (total) {
        BV_CUDA(ctx, cudaMemcpyAsync(ctx->d_rs_bases, bases, total, cudaMemcpyHostToDevice, st));
        BV_CUDA(ctx, cudaMemcpyAsync(ctx->d_rs_values, values, total * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    }
    BV_CUDA(ctx, cudaMemcpyAsync(ctx->d_rs_start, start, ((size_t)n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    BV_CUDA(ctx, cudaMemcpyAsync(ctx->d_rs_ref, ref_base, n, cudaMemcpyHostToDevice, st));
    BV_CUDA(ctx, cudaMemcpyAsync(d_mask, alt_mask, n, cudaMemcpyHostToDevice, st));
    const bool prof = ctx->profiling;
    if (prof) BV_CUDA(ctx, cudaEventRecord(ctx->ev_rs[0], st));
    const uint32_t max_grid = (uint32_t)ctx->num_sms * bv::kRsCtasPerSm;
    bv::bv_ranksum_test_kernel<<<n < max_grid ? n : max_grid, bv::kRsThreads, bv::kRsSmemBytes, st>>>(
        ctx->d_rs_bases, ctx->d_rs_values, ctx->d_rs_start, ctx->d_rs_ref, d_mask, n, ctx->d_rs_out);
    BV_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    if (prof) { BV_CUDA(ctx, cudaEventRecord(ctx->ev_rs[1], st)); ctx->ev_rs_valid = true; }
    BV_CUDA(ctx, cudaMemcpyAsync(phred_out, ctx->d_rs_out, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
    BV_CUDA(ctx, cudaStreamSynchronize(st));
    return BV_OK;
}

uint32_t bv_suggest_tile_sites(const bv_ctx* ctx, uint32_t n_samples, uint64_t max_bytes) {
    const uint64_t pitch = ((uint64_t)(n_samples ? n_samples : 1) + 15) / 16 * 16;
    uint64_t fit = max_bytes / (3 * pitch);
    if (fit < 1) fit = 1;
    if (fit > 0xffffffffull) fit = 0xffffffffull;
    const uint64_t sms = ctx && ctx->num_sms > 0 ? (uint64_t)ctx->num_sms : 148;
    const uint64_t unit = sms * (n_samples > (uint32_t)bv::kLongRowSamples ? bv::kCountWarpsLong : bv::kCountWarpsShort);
    return (uint32_t)(fit >= unit ? fit / unit * unit : fit);
}

int bv_host_alloc(void** out_ptr, size_t bytes) {
    if (!out_ptr) return set_err(nullptr, BV_ERR_ARG, "null argument");
    cudaError_t e = cudaHostAlloc(out_ptr, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) return set_err(nullptr, BV_ERR_CUDA, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    return BV_OK;
}

int bv_host_free(void* ptr) {
    cudaError_t e = cudaFreeHost(ptr);
    if (e != cudaSuccess) return set_err(nullptr, BV_ERR_CUDA, "cudaFreeHost failed: %s", cudaGetErrorString(e));
    return BV_OK;
}

}  // extern "C"
