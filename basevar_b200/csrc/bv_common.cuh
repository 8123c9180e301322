// bv_common.cuh -- definitions shared by the kernels of the basetype core (sm_100a).
//
// The per-site statistical core of `basevar basetype` runs as a sequence of small kernels, split by the KIND of work so that
// every kernel is small and all of its warps execute the same code (one fused kernel was measured instruction-cache bound:
// 59 % of its stall samples were "no instruction" with 24 warps per SM spread over 76 KB of code):
//
//   K0  bv_expand_kernel  (bv_expand_kernel.cuh)   sparse tiles only (host or device resident): the covered cells -> the dense
//        planes in HBM.
//   K1  bv_count_kernel   (bv_count_kernel.cuh)    every site, every cell: streams the base + strand planes through
//        per-warp TMA rings and counts -- per-base depths and the 2x4 strand table.  Sites whose reads all equal REF get
//        their final record here; the others get their counts and the state BV_STATE_SCALAR.
//   K2  bv_scalar_kernel  (bv_finish_kernels.cuh)  one THREAD per site in state SCALAR: active alleles, the strand-bias test
//        of the CVG row where it is closed form (else it is listed for KF); final record unless the result depends on base
//        qualities (then state BOUND or EM).
//   K3  bv_bound_kernel   (bv_finish_kernels.cuh)  one warp per site in state BOUND (REF plus one minor allele carried by
//        a few reads -- sequencing errors): fetches the row's base + qual planes and settles the LRT by a rigorous bound
//        on the likelihood ratio, without running the EM; what the bound cannot decide goes to state EM.
//   K4a bv_hist_kernel    (bv_em_kernels.cuh)      one warp per site in state EM: (base, phred) histogram of the row, compact
//        bins, one EM task per candidate subset of the active alleles.
//   K4b bv_em_task_kernel (bv_em_kernels.cuh)      one THREAD per EM task (the whole EM of one subset on the site's bins); the
//        thread that finishes a site's last task replays the LRT elimination on the results and completes the record (ALT, AF,
//        QUAL; the Fisher test of the VCF row is listed for KF).  bv_em_iter_kernel runs the iterations first when the
//        convergence test uses fabs.
//   KF  bv_fisher_kernel  (bv_finish_kernels.cuh)  the two-sided Fisher exact tests K2 and K4 listed, a pair of lanes per test
//        (one per tail), the tests over wide supports (bisection + tail sums) apart from those over narrow ones (the
//        reference's walk), so that every warp runs one path.
//   K5 / K6 (bv_call_kernels.cuh) rank sums and population-group frequencies of the called sites; K7 bv_pack_kernel
//        (bv_finish_kernels.cuh) the compact result transport; K8 bv_list_kernel (bv_list_kernel.cuh) lrt(list) per site.
//
// Work moves between the kernels through compact lists of site indices (appended with warp-aggregated atomics, so their
// order varies from run to run; every site is independent, so the records do not).  The record's `reserved0` word
// carries the site's state for inspection (0 in every finished record).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/basevar_b200.h"

namespace bv {

constexpr int kQStride = 128;                // phred slots per LUT row
constexpr int kQSlots = 96;                  // phred slots per histogram row (0..93 valid; larger values clamp to 95)
constexpr int kHistWords = 5 * kQSlots;      // (A,C,G,T,other) x phred
constexpr int kSmemBins = 160;               // compact bins kept in shared memory; more spill to global scratch
constexpr int kMaxBins = kHistWords;         // upper bound on distinct (base, phred) bins
constexpr int kLogTabEntries = 128;
constexpr int kLutOneMinusEps = 0;           // lut[0][q] = 1 - eps(q)
constexpr int kLutEpsThird = 1;              // lut[1][q] = eps(q) / 3
constexpr int kLutLogMatch = 2;              // lut[2][q] = log(1 - eps(q))   (glibc)
constexpr int kLutLogMis = 3;                // lut[3][q] = log(eps(q) / 3)   (glibc)
constexpr uint32_t kFull = 0xffffffffu;

constexpr uint32_t kStateDone = 0;           // record is final
constexpr uint32_t kStateScalar = 1;         // counts are final, K2 has to finish the record
constexpr uint32_t kStateBound = 2;          // result depends on base qualities; K3 tries the likelihood-ratio bound
constexpr uint32_t kStateEM = 3;             // result depends on base qualities; K4 runs EM + LRT

constexpr int kCntSlow = 0, kCntBound = 1, kCntEm = 2;                    // SiteKernelArgs::counters (10 is unused)
constexpr int kCntListPairs = 3;                                          // chunk ticket of bv_list_pairs_kernel (bv_list_kernel.cuh)
constexpr int kCntCalled = 4, kCntGroupNext = 5;                          // called sites (K4 -> K5, K6)
constexpr int kCntBadCell = 6;                                            // malformed sparse input (K0, bv_expand_kernel.cuh)
constexpr int kCntEmHdr = 7, kCntEmPool = 8;                              // K4a -> K4b: EM sites and the pool of their bins
constexpr int kCntEmTask2 = 9, kCntEmTask3 = 11, kCntEmTask4 = 12;        // EM tasks by number of alleles in the candidate subset
constexpr int kCntFull = 13;                                              // full records of a compact tile (bv_pack_kernel)
constexpr int kCntFisherNarrow = 14, kCntFisherWide = 15;                   // queued Fisher tests (K2, K4b -> bv_fisher_kernel)
constexpr int kCntEmFetch2 = 16, kCntEmFetch3 = 17, kCntEmFetch4 = 18;      // next task of each list (bv_em_iter_kernel)
constexpr int kNumCounters = 24;

// word indices of bv_site_out seen as 32 x u32
constexpr int kWDepth = 0, kWOther = 4, kWState = 5, kWFwd = 6, kWRev = 10, kWAlt = 14, kWInfo = 15;

// One site of the EM list after K4a (bv_em_kernels.cuh): its compact (base, phred) bins in the pool, its EM tasks.
struct __align__(16) EmSiteHdr {
    uint32_t site;
    uint32_t bins_off;       // first word of the site's bins in SiteKernelArgs::em_pool
    uint32_t nb;             // number of bins
    uint32_t act_flags;      // active alleles before the LRT (bits 0-3) | BV_FLAG_* raised so far << 8 | bit 16 + b: the EM of the
                             // single-allele model {b} raises BV_FLAG_EM_MAXITER (single_em_flag; none at the default parameters)
    uint32_t task[3];        // slot of the site's first task among the 2-, 3- and 4-allele tasks (em_tasks / em_res)
    uint32_t remaining;      // tasks not finished yet: the thread that takes it to 0 decides the site
    uint32_t depth[4];
    uint32_t total;          // depth[0..3] + depth_other
    uint32_t base_start[3];  // bins are sorted by base: A = [0, s0), C = [s0, s1), G = [s1, s2), T = [s2, s3), other = [s3, nb);
                             // base_start[0] = s0 | s1 << 16, base_start[1] = s2 | s3 << 16, base_start[2] unused
};
static_assert(sizeof(EmSiteHdr) == 64, "EmSiteHdr layout");
constexpr int kEmResDoubles = 10;            // per EM task: log-likelihood, f[4], flags (as bits of a u64); between bv_em_iter_kernel
                                             // and bv_em_task_kernel: f[k], fp[k] (k-th allele of the subset) in [0..3], [4..7], flags in [8]
constexpr uint32_t kEmTaskInvalid = 0xffffffffu;
constexpr uint32_t kFisherVcfRow = 1u << 24;   // list_fisher entry: the test of the VCF row (ref vs called ALT), else that of the CVG row
constexpr uint32_t kFisherWide = 1u << 25;     // (in the queues of a CTA only) the table's support is wider than kFisherNarrowSupport

struct SiteKernelArgs {
    const uint8_t* base;
    const uint8_t* qual;
    const uint8_t* strand;
    const uint8_t* ref_base;
    bv_site_out* out;
    const double* lut;       // [4][kQStride]
    const double2* logtab;   // [kLogTabEntries] {1 / c, -log(1 / c)}, c = 1 + (i + 1/2) / 128: log_tab() of bv_em_kernels.cuh
    const double* logfact;   // [max_samples + 2], lgamma(k+1) from glibc
    uint32_t* bin_spill;     // [K4 warps][kMaxBins] global copy of the compact bins (used when > kSmemBins)
    double* lml_spill;       // [K4 warps][kMaxBins] per-bin EM state for the same case
    uint32_t* list_slow;     // work lists (site indices), each with room for n_sites entries: K1 -> K2,
    uint32_t* list_bound;    //   K2 -> K3,
    uint32_t* list_em;       //   K2 and K3 -> K4
    uint32_t* list_fisher;   //   K2 and K4b -> bv_fisher_kernel: [2 * n_sites] queued Fisher tests (site | kFisherVcfRow), those over narrow
                             //   supports from the front, those over wide supports from the back
    uint32_t* counters;      // [kNumCounters], zeroed before K1
    // K4a -> K4b (bv_em_kernels.cuh)
    EmSiteHdr* em_hdr;       // [n_sites]
    uint32_t* em_pool;       // [n_sites][kMaxBins] compact bins of the EM sites, allocated with kCntEmPool
    uint32_t* em_tasks;      // hdr index | subset << 28; three lists one after the other: 2-, 3- and 4-allele subsets,
                             // em_task_cap[k] slots each (6 / 4 / 1 per site), allocated with kCntEmTask2 / 3 / 4
    double* em_res;          // [sum of em_task_cap][kEmResDoubles], indexed like em_tasks
    double* em_single;       // [n_sites][4], indexed like em_hdr: log-likelihood of the single-allele model of each ACTIVE base
    uint32_t em_task_cap[3];
    // compact record transport (BV_OUT_COMPACT): null unless the tile asked for it
    uint32_t em_resume;      // bv_em_task_kernel: the EM iterations were run by bv_em_iter_kernel, start from its frequencies
    uint32_t em_task_split;  // tiles with more EM tasks than this run bv_em_task_kernel<kTaskHiCtas>, the others <kTaskLoCtas>
    uint2* brief;            // [n_sites] device copy of the briefs: K1 writes them, bv_pack_kernel completes them
    bv_site_out* full_out;   // the full records, written by bv_pack_kernel: pinned host memory (mapped) of a slot, or the device
                             // buffer of a device-resident tile (bv_device_out::d_full)
    // called sites (n_alt > 0): rank sums (K5) and population-group frequencies (K6); all null / 0 when not asked for
    uint32_t* list_called;   // K4 -> K5, K6: site indices, room for n_sites entries
    const uint8_t* mapq;     // [n_sites][aux_pitch]
    const uint16_t* rpr;     // [n_sites][rpr_pitch] (elements)
    uint64_t aux_pitch;
    uint64_t rpr_pitch;
    const uint8_t* sample_group;   // [round16(n_samples)] group index per sample, BV_GROUP_NONE padding
    bv_call_out* calls;      // [n called sites], entry k belongs to list_called[k]
    bv_group_out* groups;    // [n called sites][n_groups]
    uint32_t n_groups;
    uint32_t pad0;
    uint64_t pitch;          // bytes between rows of the base and strand planes
    uint64_t qual_pitch;     // bytes between rows of the qual plane (it may live in pinned host memory, see bv_tile_submit)
    uint32_t n_sites;
    uint32_t n_samples;
    double min_af;           // (double)(float)min_af
    double em_eps;           // (double)(float)0.001
    double lrt_threshold;
    int em_max_iter;
    int abs_mode;
};

// Dynamic shared memory of K1 and K3.  Device functions reach it through accessors (not through pointer arguments) so
// that the compiler knows the address space and emits LDS/STS/ATOMS.
extern __shared__ __align__(128) unsigned char bv_smem_raw[];

// REF character -> base code 0..3, or -1 (toupper first: src/basetype.cpp:171)
__device__ __forceinline__ int ref_code_of(uint32_t rc) {
    if (rc >= 'a' && rc <= 'z') rc -= 32;
    return rc == 'A' ? 0 : rc == 'C' ? 1 : rc == 'G' ? 2 : rc == 'T' ? 3 : -1;
}

// ---- TMA bulk copies + mbarrier (sm_90+; SASS UBLKCP / SYNCS) -----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// ---- programmatic dependent launch (griddepcontrol, sm_90+) along K2 -> K3 -> ... -> KF (launch_site_kernel, bv_api.cu) ------
// K3..KF are launched with programmatic stream serialization: a kernel's CTAs may start while the kernel before it still
// runs, once every CTA of that kernel has called grid_dep_launch (or exited).  Everything a kernel reads that an earlier
// kernel of the tile wrote (counters, work lists, records, the EM tables) comes after grid_dep_wait, which returns once
// the kernel before has completed and its writes are visible; every CTA calls it, also those with no work, so that a
// kernel never completes before the one it follows.  Both are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// valid = number of real cells in this 16-cell vector (>= 16 for all but the row's last vector): padding cells
// are turned into 'N'
__device__ __forceinline__ void mask_tail(uint4& vb, int valid) {
    uint32_t w[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int left = valid - 4 * k;
        const uint32_t keep = left >= 4 ? 0xffffffffu : (left <= 0 ? 0u : (0xffffffffu >> (8 * (4 - left))));
        w[k] = (w[k] & keep) | (0x05050505u & ~keep);
    }
    vb = make_uint4(w[0], w[1], w[2], w[3]);
}

// exact `(double)dep / (double)total >= min_af` (src/basetype.cpp:137) with the trivial cases short-cut
__device__ __forceinline__ bool is_active(uint32_t dep, uint32_t total, double dtot, double min_af) {
    if (dep == 0) return 0.0 >= min_af;
    if (dep == total) return 1.0 >= min_af;
    // away from the boundary the product decides (one multiply instead of a division); within 1e-9 of it, the
    // reference's own expression
    const double thr = min_af * dtot, x = (double)dep;
    if (x > thr * 1.000000001) return true;
    if (x < thr * 0.999999999) return false;
    return x / dtot >= min_af;
}

// BV_FLAG_EM_MAXITER of the EM of a single-allele model {b} that starts from f_b = d / total (0 < d <= total), the closed form
// of its loop count (src/algorithm.h:210-255): the first M-step sets f_b = 1 exactly, so in the loop's first iteration every
// log marginal moves by -log(d / total) and in every later one by 0.  The loop therefore ends after one iteration when that
// first sum is below eps, after two when 0 < eps, and otherwise runs all em_max_iter.  (A phred-0 read of b makes the
// marginals NaN; that loop count is not modelled, see BV_FLAG_EM_MAXITER in the header.)
// Out of line: the kernels that call it run at the default parameters, where the answer is 0 without it.
__device__ __noinline__ uint32_t single_em_flag_off_default(uint32_t d, uint32_t total, int max_iter, double eps, int abs_mode) {
    if (max_iter <= 1) return BV_FLAG_EM_MAXITER;
    double delta1 = 0.0;
    if (d != total) {
        const double lg = -log((double)d / (double)total);
        delta1 = (double)total * (abs_mode == BV_EM_ABS_INT_TRUNC ? (double)(int)lg : lg);
    }
    const bool flag = !(delta1 < eps) && (max_iter == 2 || !(eps > 0.0));
    return flag ? BV_FLAG_EM_MAXITER : 0u;
}
__device__ __forceinline__ uint32_t single_em_flag(uint32_t d, uint32_t total, const SiteKernelArgs& a) {
    if (a.em_max_iter > 2 && a.em_eps > 0.0) return 0u;   // the defaults: done after at most two iterations
    return single_em_flag_off_default(d, total, a.em_max_iter, a.em_eps, a.abs_mode);
}
// At em_max_iter 0 the EM reports the first E-step's log marginals, L * f0 with f0 = d / total: the closed form of the
// single-allele log-likelihood (f = 1) plus this.  Out of line for the same reason.
__device__ __noinline__ double first_estep_ll_shift(uint32_t d, double dtot) { return dtot * log((double)d / dtot); }

__device__ __forceinline__ uint32_t sel4u(int j, uint32_t v0, uint32_t v1, uint32_t v2, uint32_t v3) {
    return j == 0 ? v0 : j == 1 ? v1 : j == 2 ? v2 : v3;
}

}  // namespace bv
