// bv_em_kernels.cuh -- K4: the sites whose result depends on base qualities (state kStateEM): K4a bv_hist_kernel, K4b bv_em_task_kernel
// (+ bv_em_iter_kernel when the EM's convergence test uses fabs).
//
// The reference runs, per such site, one EM over the full active set and then backward elimination: for every
// (n-1)-subset of the n active alleles another EM, keep the best, stop when 2 dLL >= 24 (BaseType::lrt,
// src/basetype.cpp:130-199; _f, :105-128; EM, src/algorithm.h:210-255).  The EMs of one site are independent of each
// other -- only WHICH of them the elimination consults depends on earlier results -- and one EM is a short serial
// recurrence over the site's non-empty (base, phred) bins.  So the work is split by its shape:
//
//   K4a bv_hist_kernel     one WARP per site: streams the row's base + qual planes (TMA ring), (base, phred) histogram in
//                          shared memory, compaction to bins.  A site with one active allele is finished here (closed
//                          form).  A site with >= 2 gets a header, its bins in a pool, and one EM TASK per subset of
//                          >= 2 active alleles (1, 4 or 11 tasks for 2, 3 or 4 active alleles; single-allele models are
//                          closed form), listed by subset size.
//   K4b bv_em_task_kernel  one THREAD per task: the whole EM of one candidate subset over the site's bins, staged in shared
//                          memory.  No warp-wide repetition of scalar work, every lane of the FP64 pipe carries a different
//                          EM.  (A tile with few tasks would leave the GPU idle behind their serial chains: it gets four
//                          lanes per task; the sums are formed in the same order either way.)
//                          The thread that stores the LAST result of a site then decides it: replays the elimination
//                          loop on the table of task results (first-minimum argmin in the reference's subset order,
//                          threshold, flags), ALT / AF / QUAL (chi-square survival function) -- scalar work that overlaps
//                          with the EMs of other warps.  The strand-bias Fisher test of the VCF row is only listed here;
//                          bv_fisher_kernel (bv_finish_kernels.cuh) runs the listed tests of a tile together.
//
// At most 3 of the 11 tasks of a 4-allele site are never consulted (the elimination needs <= 8 EMs); evaluating them
// anyway removes every dependency between EMs.  A flag an unconsulted task raises (BV_FLAG_EM_MAXITER) is not reported.
// Scratch (headers, bin pool, task lists, results) has room for every site of the largest tile to be an EM site with kMaxBins
// bins and all 11 tasks (scratch_reserve, bv_api.cu), so every EM site of every tile takes this one path: its records do not
// depend on the context's max_sites nor on the order in which K4a's warps allocate.  (A fallback that finished the sites that
// did not fit inside K4a with lrt_on_bins associated its sums differently: AF / QUAL / chi2 then differed in the last bits
// between a small and a large context, and from run to run.)
#pragma once
#include "bv_finish_kernels.cuh"

namespace bv {

// ---- K4a: one site in state kStateEM -----------------------------------------------------------------------------------------
// Everything here is warp-uniform.  The record (counts, FS of the CVG row, flags, active set) comes from K1 / K2.
template <bool LONG>
__device__ __noinline__ void hist_site(uint32_t site) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const int lane = threadIdx.x & 31;
    if (lane < 8) reinterpret_cast<uint4*>(&W.rec)[lane] = reinterpret_cast<const uint4*>(cs.a.out + site)[lane];
    __syncwarp();
    const uint32_t d0 = W.rec.depth[0], d1 = W.rec.depth[1], d2 = W.rec.depth[2], d3 = W.rec.depth[3];
    const uint32_t total = d0 + d1 + d2 + d3 + W.rec.depth_other;
    // ---- lrt (src/basetype.cpp:130-199): the active set (total > 0 here) was worked out by K2 ----
    const uint32_t act = (reinterpret_cast<const uint32_t*>(&W.rec)[kWAlt] >> 8) & 0xfu;
    if (lane == 0) W.flag_word = W.rec.flags;
    __syncwarp();

    // histogram the row by (base, phred)
    const uint32_t h = LONG ? build_hist_long(site) : build_hist(site, nullptr, 0);
    const uint32_t qmin = h & 0xffu, qmax = (h >> 8) & 0xffu;
    if (lane == 0) W.flag_word |= h >> 16;
    __syncwarp();
    if (__popc(act) >= 2) {
        const int nb = compact_bins(qmin, qmax);
        // ---- hand the site to K4b: bins into the pool, one task per subset of >= 2 active alleles ----
        // lane m < 16 looks after subset m; tasks are listed by subset size (2, 3, 4 alleles), in ascending subset order
        const uint32_t m = (uint32_t)lane;
        const int k = __popc(m);
        const bool is_task = lane < 16 && (m & ~act) == 0u && k >= 2;
        const uint32_t bal2 = __ballot_sync(kFull, is_task && k == 2), bal3 = __ballot_sync(kFull, is_task && k == 3),
                       bal4 = __ballot_sync(kFull, is_task && k == 4);
        const uint32_t n_k[3] = {(uint32_t)__popc(bal2), (uint32_t)__popc(bal3), (uint32_t)__popc(bal4)};
        // five allocations at once: pool (lane 0), header (lane 1), task slots of each size (lanes 2-4).  They cannot fail: the
        // scratch has kMaxBins pool entries, one header and 6 / 4 / 1 task slots per site of the tile (scratch_reserve).
        uint32_t got = 0, want = 0;
        if (lane == 0) want = (uint32_t)nb;
        if (lane == 1) want = 1u;
        if (lane >= 2 && lane < 5) want = n_k[lane - 2];
        constexpr int kCnt[5] = {kCntEmPool, kCntEmHdr, kCntEmTask2, kCntEmTask3, kCntEmTask4};
        if (lane < 5 && want) got = atomicAdd(cs.a.counters + kCnt[lane], want);
        const uint32_t off = __shfl_sync(kFull, got, 0), hdr = __shfl_sync(kFull, got, 1);
        const uint32_t t2 = __shfl_sync(kFull, got, 2), t3 = __shfl_sync(kFull, got, 3), t4 = __shfl_sync(kFull, got, 4);
        const uint32_t base3 = cs.a.em_task_cap[0], base4 = base3 + cs.a.em_task_cap[1];
        if (is_task) {
            const uint32_t my_t = k == 2 ? t2 + (uint32_t)__popc(bal2 & ((1u << lane) - 1u))
                                : k == 3 ? base3 + t3 + (uint32_t)__popc(bal3 & ((1u << lane) - 1u)) : base4 + t4;
            cs.a.em_tasks[my_t] = hdr | (m << 28);
        }
        const uint32_t* bins = nb <= kSmemBins ? W.bins : cs.a.bin_spill + (size_t)(blockIdx.x * kQualWarps + (threadIdx.x >> 5)) * kMaxBins;
        for (int i = lane; i < nb; i += 32) cs.a.em_pool[off + i] = bins[i];
        // first bin of each base (bins are sorted by base): lane b counts the bins of bases < b + 1
        uint32_t below = 0;
        for (int i = lane; i < nb; i += 32) {
            const uint32_t b = bin_base(bins[i]);
            below += (b < 1u) | ((uint32_t)(b < 2u) << 8) | ((uint32_t)(b < 3u) << 16) | ((uint32_t)(b < 4u) << 24);
        }
        // (a lane sees at most kMaxBins / 32 = 15 bins, so the four byte counters cannot overflow before the reduction)
        const uint32_t s0 = __reduce_add_sync(kFull, below & 0xffu), s1 = __reduce_add_sync(kFull, (below >> 8) & 0xffu),
                       s2 = __reduce_add_sync(kFull, (below >> 16) & 0xffu), s3 = __reduce_add_sync(kFull, below >> 24);
        // log-likelihoods of the four single-allele models (closed form, see single_allele_ll): the last elimination round of
        // the site's decision consults two of them
        {
            double sl[4];
            single_allele_ll4(bins, nb, sl);
            if (lane < 4) cs.a.em_single[(size_t)hdr * 4 + lane] = lane == 0 ? sl[0] : lane == 1 ? sl[1] : lane == 2 ? sl[2] : sl[3];
        }
        if (lane == 0) {
            uint4 w0, w1, w2, w3;
            w0.x = site; w0.y = off; w0.z = (uint32_t)nb; w0.w = act | (W.flag_word << 8);
            w1.x = t2; w1.y = base3 + t3; w1.z = base4 + t4; w1.w = n_k[0] + n_k[1] + n_k[2];
            w2.x = d0; w2.y = d1; w2.z = d2; w2.w = d3;
            w3.x = total; w3.y = s0 | (s1 << 16); w3.z = s2 | (s3 << 16); w3.w = 0;
            uint4* H = reinterpret_cast<uint4*>(cs.a.em_hdr + hdr);
            H[0] = w0; H[1] = w1; H[2] = w2; H[3] = w3;
        }
        __syncwarp();
        return;   // the record is completed by K4b
    }
    // One active allele: the reference still runs one EM; its answer is closed form (see single_allele_ll):
    // AF == 1.0 exactly, or NaN when a phred-0 read of that base exists.
    {
        const int b = __ffs(act) - 1;
        const bool bad = qmin == 0 && W.hist[b * kQSlots] != 0;
        const double v = bad ? __longlong_as_double(0x7ff8000000000000ll) : 1.0;
        __syncwarp();
        if (lane < 4) W.res_f[lane] = lane == b ? v : 0.0;
        if (qmin <= qmax) {   // histogram back to zero
#pragma unroll 1
            for (uint32_t q = qmin + lane; q <= qmax; q += 32) {
#pragma unroll
                for (int r = 0; r < 5; ++r) W.hist[r * kQSlots + q] = 0;
            }
        }
    }
    __syncwarp();
    uint32_t flags = W.flag_word;

    // ---- ALT / QUAL (src/basetype.cpp:170-196) ----
    // Here only the rule that needs no arithmetic (mono-allelic 5000); the chi-square survival function and the Fisher
    // test of the VCF row are scalar work: the site is queued and vcf_flush() does them one thread per site (the test itself:
    // bv_fisher_kernel).
    const int ref_code = ref_code_of(cs.a.ref_base[site]);
    const uint32_t ref_bit = ref_code >= 0 ? (1u << ref_code) : 0u;
    const uint32_t alt_set = act & ~ref_bit;
    const int n_alt = __popc(alt_set);
    double qual = 0.0;
    if (n_alt) {
        const int first_act = __ffs(act) - 1;
        const double r = (double)sel4u(first_act, d0, d1, d2, d3) / (double)total;
        if (total > 10 && r > 0.5) { qual = 5000.0; flags |= BV_FLAG_MONO_QUAL; }
    }

    // ---- record ----
    __syncwarp();
    if (lane == 0) {
        bv_site_out& r = W.rec;
        r.reserved0 = kStateDone;
        // ALT alleles in ACGT order of the active set (src/basetype.cpp:172-177)
        uint32_t alts = 0;
        int k = 0;
        const double af[4] = {W.res_f[0], W.res_f[1], W.res_f[2], W.res_f[3]};
        r.af[0] = 0.0; r.af[1] = 0.0; r.af[2] = 0.0; r.af[3] = 0.0;
        if (alt_set & 1) { r.af[k] = af[0]; alts |= 0u << (8 * k); ++k; }
        if (alt_set & 2) { r.af[k] = af[1]; alts |= 1u << (8 * k); ++k; }
        if (alt_set & 4) { r.af[k] = af[2]; alts |= 2u << (8 * k); ++k; }
        if (alt_set & 8) { r.af[k] = af[3]; alts |= 3u << (8 * k); ++k; }
        r.n_alt = (uint8_t)n_alt;
        r.alt[0] = (uint8_t)alts; r.alt[1] = (uint8_t)(alts >> 8); r.alt[2] = (uint8_t)(alts >> 16); r.alt[3] = (uint8_t)(alts >> 24);
        r.n_active = 1;
        r.flags = (uint8_t)flags;
        r.em_calls = 1;
        r.qual = qual;
        r.chi2 = 0.0;
        r.fs_vcf = 0.0;
        // called sites go on to the rank-sum / population-group kernels (bv_call_kernels.cuh)
        if (n_alt && cs.a.list_called) cs.a.list_called[atomicAdd(cs.a.counters + kCntCalled, 1u)] = site;
        if (n_alt) W.vcf_site[W.vcf_n++] = site;
    }
    __syncwarp();
    if (lane < 8) reinterpret_cast<uint4*>(cs.a.out + site)[lane] = reinterpret_cast<const uint4*>(&W.rec)[lane];
    __syncwarp();   // also orders the record's stores before vcf_flush() reads them from other lanes
    if (W.vcf_n == 32) vcf_flush();
}

// Persistent warps over the EM list.  LONG: the shape for rows of more than kLongRowSamples
// samples (kLongWarps warps per CTA, build_hist_long).
template <bool LONG>
__global__ void __launch_bounds__((LONG ? kLongWarps : kQualWarps) * 32, 1) bv_hist_kernel(const __grid_constant__ SiteKernelArgs a) {
    QualCta& cs = cta_shared();
    QualWarp& W = warp_smem();
    const int lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < 4 * kQStride; i += blockDim.x) cs.lut[i] = a.lut[i];
    if (threadIdx.x == 0) cs.a = a;
    for (int i = lane; i < kHistWords; i += 32) W.hist[i] = 0;
    if (lane == 0) {
        W.flag_word = 0;
        W.p2_phase = 0;
        W.vcf_n = 0;
        for (int b = 0; b < kP2Bufs; ++b) mbar_init(&W.p2bar[b], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    grid_dep_wait();
    // The EM list is final (K3 is done).  A site costs one pass over its row, the same for every site of a tile, so the sites
    // are dealt out statically -- entry i to warp i mod (all warps), neighbours in the list to different SMs -- and the next
    // entry is read while this one is worked on.  (A shared fetch counter cost every site a round trip to one L2 address that
    // 4,736 warps queue on: 17 % of the kernel's stall samples on deep pileups.)
    const uint32_t n_em = a.counters[kCntEm];
    const uint32_t total_warps = gridDim.x * (blockDim.x >> 5);
    uint32_t i = (threadIdx.x >> 5) * gridDim.x + blockIdx.x;
    uint32_t site_next = i < n_em ? a.list_em[i] : 0u;
    for (; i < n_em; i += total_warps) {
        const uint32_t site = site_next;
        if (i + total_warps < n_em) site_next = a.list_em[i + total_warps];
        hist_site<LONG>(site);
    }
    grid_dep_launch();
    if (W.vcf_n) vcf_flush();
}

// =====================================================================================================================
// K4b: one thread per EM task; the thread that finishes a site's last task decides the site.
// =====================================================================================================================
constexpr int kTaskThreads = 128;
constexpr int kTaskLoCtas = 3;                     // resident CTAs per SM the two builds of bv_em_task_kernel are compiled for: tiles with few EM tasks ...
constexpr int kTaskHiCtas = 4;                     // ... and tiles with many
static_assert(kTaskLoCtas != kTaskHiCtas, "the two builds of bv_em_task_kernel are told apart by their CTA count");
constexpr int kStageBins = 96;                     // bins per site staged in shared memory; longer lists are read from the pool
constexpr int kStageStride = kStageBins + 1;       // odd: the rows of 32 different sites start in 32 different banks
constexpr uint32_t kG4MaxTasks = 12288;            // tiles with at most this many EM tasks give each task four lanes

struct __align__(16) TaskCta {
    double lut[4][kQSlots];           // 1 - eps(q), eps(q) / 3, log(1 - eps(q)), log(eps(q) / 3)
    double2 ltab[kLogTabEntries];     // log_tab()'s table
    uint32_t n_decide;                // sites whose last task finished in this round of the CTA ...
    uint32_t decide_hdr[kTaskThreads];   // ... their headers: decided one thread per site after the round
    uint32_t n_fs;                    // Fisher tests of the VCF rows of decided sites, listed by decide_site ...
    uint32_t fs_site[2 * kTaskThreads];  // ... on their way to list_fisher, a CTA of them at a time
    uint32_t bins[kTaskThreads * kStageStride];   // one row per task of the round
};
constexpr size_t kTaskSmemBytes = sizeof(TaskCta);
static_assert(kTaskSmemBytes <= 232448, "shared memory of the EM task kernel exceeds 227 KB");

// The G lanes (1 or 4, aligned) that share one task.  Sums over the bins of a task are ALWAYS formed the same way, whatever G
// is: four partial sums over the visits u = 0, 1, 2, 3 (mod 4), combined as (p0 + p2) + (p1 + p3).  One lane keeps the four
// partial sums itself (four independent FP64 chains); four lanes keep one each and combine them with two butterfly steps,
// which form exactly that expression.  The records therefore do not depend on how many lanes a launch gave its tasks
// (i.e. on how many tasks the tile had).
struct LaneGroup {
    int G, gl;
    uint32_t mask;
    __device__ __forceinline__ double sum4(double v) const {   // G == 4: every lane of the group gets (p0 + p2) + (p1 + p3)
        v += __shfl_xor_sync(mask, v, 2);
        v += __shfl_xor_sync(mask, v, 1);
        return v;
    }
    __device__ __forceinline__ bool any(bool p) const { return (__ballot_sync(mask, p) & mask) != 0u; }
};
__device__ __forceinline__ double sum4(const double (&p)[4]) { return (p[0] + p[2]) + (p[1] + p[3]); }

// log(r) for the ratio of two marginals of consecutive E-steps: once the EM settles r is within 2^-10 of 1 for every bin,
// and t - t^2/2 + t^3/3 - t^4/4 (t = r - 1, exact) is then good to 2e-16 of t -- below the rounding of a full logarithm,
// which costs ten times as many instructions.  The sum these terms go into is only compared with 0.001.
__device__ __forceinline__ double log_ratio(double r) {
    const double t = r - 1.0;
    if (fabs(t) < 0.0009765625) return t * fma(t, fma(t, fma(t, -0.25, 1.0 / 3.0), -0.5), 1.0);
    return log(r);
}

// log(x) through a 128-entry table: x = 2^e * z, z in [1, 2); the top seven mantissa bits pick c = 1 + (i + 1/2) / 128 with
// tab[i] = {1 / c rounded, -log(1 / c rounded)} (glibc, bv_api.cu), r = z / c - 1 is exact in one fma and |r| < 2^-8, so
// log(1 + r) is six terms of its series (the next one is below 3e-18).  Absolute error <= 2.8e-16 * max(|log x|, ln 2) against 80-bit
// logl on 2e7 arguments (tools/log_tab_check.c, tests/test_log_tab_cpu.py; libdevice: 1.1e-16 * |log x|) -- every term of the EM's
// log-likelihood sums has the same sign, so the sums keep that relative error: 1e-10 on the chi-square of a 10,000-read row, whose
// check allows 1e-8 -- at a third of libdevice's instructions and WITHOUT A BRANCH: the four bins a thread works on side by side
// stay one straight-line block (no divergence regions between them) for the scheduler to overlap.  Zero, denormal, negative, inf and NaN
// arguments raise `bad` (the value returned for them means nothing); the caller then forms its sum again with the library
// function (em_sum_slow).
__device__ __forceinline__ double log_tab(double x, const double2* tab, uint32_t& bad) {
    const uint32_t hi = (uint32_t)__double2hiint(x);
    bad |= (hi - 0x00100000u >= 0x7fe00000u) ? 1u : 0u;
    const double2 t = tab[(hi >> 13) & 0x7fu];
    const double z = __hiloint2double((int)((hi & 0x000fffffu) | 0x3ff00000u), __double2loint(x));
    const double r = fma(z, t.x, -1.0);
    double p = fma(r, -1.0 / 6.0, 0.2);
    p = fma(r, p, -0.25);
    p = fma(r, p, 1.0 / 3.0);
    p = fma(r, p, -0.5);
    p = fma(r * r, p, r);
    return fma((double)((int)(hi >> 20) - 1023), 0.693147180559945309417, t.y) + p;
}

// The bins of a site are sorted by base, so the bins of allele j[k] of a candidate subset are one RUN [r0[k], r1[k]) of the list.
// Inside run k every bin has the likelihood row {e3, ..., 1 - eps at k, ..., e3}: its marginal is
//     m = (1 - eps) * f_k + e3 * fo_k,        fo_k = the sum of the subset's OTHER frequencies (A, C, G, T order),
// (for two alleles exactly the reference's lik * freq sum, src/algorithm.h:160-172), and with w = c / m its posteriors add
// w * (1 - eps) * f_k to column k and w * e3 * f_j to every other column j.  Two sums per run are therefore enough,
//     o_k = sum of w * (1 - eps),    a_k = sum of w * e3        (all terms positive: nothing cancels),
// and the M-step's column sums are s_j = f_j * (o_j + sum of a_k over the other runs k): ten FP64 instructions and two
// accumulators per bin, whatever the number of alleles (one multiply-add per allele, twice, and NA accumulators before).
// A bin whose base is OUTSIDE the subset (another allele, or the "other" class) has the row {e3, e3, ...}: marginal e3 * F
// (F = sum of the subset's frequencies), posteriors f_j / F whatever its phred.  All such bins together add c_out * f_j / F
// -- one term instead of a pass over them -- and only the bins of the subset's own bases are visited.
template <int NA>
__device__ __forceinline__ double pick(const double (&v)[NA], int k) {
    double x = v[0];
#pragma unroll
    for (int i = 1; i < NA; ++i) x = k == i ? v[i] : x;
    return x;
}
template <int NA>
__device__ __forceinline__ int pick(const int (&v)[NA], int k) {
    int x = v[0];
#pragma unroll
    for (int i = 1; i < NA; ++i) x = k == i ? v[i] : x;
    return x;
}
template <int NA>
__device__ __forceinline__ void put(double (&v)[NA], int k, double x) {
#pragma unroll
    for (int i = 0; i < NA; ++i) v[i] = k == i ? x : v[i];
}
// sum of v[i], i != k, in ascending i (the skipped entry adds an exact +0.0)
template <int NA>
__device__ __forceinline__ double sum_others(const double (&v)[NA], int k) {
    double x = k == 0 ? 0.0 : v[0];
#pragma unroll
    for (int i = 1; i < NA; ++i) x += k == i ? 0.0 : v[i];
    return x;
}

// The state of one EM: the subset's alleles, the runs of their bins, the frequencies of this and of the previous E-step.
template <int NA>
struct EmState {
    int r0[NA], r1[NA];   // run of the bins of the subset's k-th allele
    double f[NA], fp[NA];
    double total;
    double c_out;         // reads outside the subset's bases
};

// One bin of a run under (fk, fo) = (frequency of the run's allele, sum of the others); (fpk, fpo) the same under the previous
// frequencies.  What x collects besides the posterior sums depends on MODE:
//   kPassDelta  c * |log m - log mp|, mp the marginal under the previous frequencies -- EM()'s convergence sum with fabs
//               (src/algorithm.h:238-250, BV_EM_ABS_DOUBLE), as one logarithm of the ratio mp / m;
//   kPassLL     c * log m: the log-likelihood _f() reports (src/basetype.cpp:119-120) is the one under the frequencies of the
//               EM's LAST E-step, and whether an E-step is the last is known before it starts (see em_task), so the sum rides
//               along with that pass instead of costing one more.
// Posterior weights are c * (1 / m) with a Newton reciprocal.  No branches: see log_tab.
constexpr int kPassPlain = 0, kPassDelta = 1, kPassLL = 2;
template <int MODE>
__device__ __forceinline__ void em_bin(uint32_t p, const double* lut, const double2* ltab, double fk, double fo, double fpk, double fpo,
                                       double& o, double& a, double& x, uint32_t& bad) {
    const uint32_t q = bin_qual(p);
    const double cd = (double)bin_count(p);
    const double ome = lut[kLutOneMinusEps * kQSlots + q], e3 = lut[kLutEpsThird * kQSlots + q];
    const double m = ome * fk + e3 * fo;
    const double inv = rcp_fast(m);
    const double w = cd * inv;
    o = fma(w, ome, o);
    a = fma(w, e3, a);
    if (MODE == kPassDelta) {
        const double mp = ome * fpk + e3 * fpo;
        x += cd * fabs(log_tab(mp * inv, ltab, bad));
    }
    if (MODE == kPassLL) x += cd * log_tab(m, ltab, bad);
}

// The sum x of a pass once more, with the library logarithm, for the EMs whose marginals left the normal range (a phred-0
// read of an allele that has all the frequency: marginal 0, everything NaN from there on as in the reference).
template <int NA, int MODE>
__device__ __noinline__ double em_sum_slow(const uint32_t* bins, const EmState<NA>& S, const double* lut, const LaneGroup& lg) {
    double xl[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 1
    for (int k = 0; k < NA; ++k) {
        const double fk = pick<NA>(S.f, k), fo = sum_others<NA>(S.f, k), fpk = pick<NA>(S.fp, k), fpo = sum_others<NA>(S.fp, k);
        const int r0 = pick<NA>(S.r0, k), r1 = pick<NA>(S.r1, k);
#pragma unroll 1
        for (int u = r0 + lg.gl; u < r1; u += lg.G) {
            const uint32_t p = bins[u];
            const uint32_t q = bin_qual(p);
            const double ome = lut[kLutOneMinusEps * kQSlots + q], e3 = lut[kLutEpsThird * kQSlots + q];
            const double m = ome * fk + e3 * fo;
            const double t = MODE == kPassLL ? nlog(m) : fabs(nlog(m) - nlog(ome * fpk + e3 * fpo));
            const double v = (double)bin_count(p) * t;
            const int slot = lg.G == 1 ? ((u - r0) & 3) : 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) xl[i] += i == slot ? v : 0.0;
        }
    }
    return lg.G == 1 ? sum4(xl) : lg.sum4(xl[0]);
}

// One E-step + M-step (src/algorithm.h:148-198) for a subset of NA alleles under frequencies S.f: s[] = the column sums of the
// posteriors.  Returns the sum x of em_bin (over the subset's own bins; kPassDelta: also the term of the bins outside).  Sums over
// the bins of a run are ALWAYS formed the same way, whatever G is (see LaneGroup): visit i of the run goes to partial sum i mod 4.
template <int NA, int MODE>
__device__ __forceinline__ double em_pass(const uint32_t* bins, const EmState<NA>& S, const double* lut, const double2* ltab,
                                          double (&s)[NA], const LaneGroup& lg) {
    constexpr bool DELTA = MODE == kPassDelta;
    double o_run[NA], a_run[NA];
    double xl[4] = {0.0, 0.0, 0.0, 0.0};
    uint32_t bad = 0;
#pragma unroll 1
    for (int k = 0; k < NA; ++k) {
        const double fk = pick<NA>(S.f, k), fo = sum_others<NA>(S.f, k);
        const double fpk = DELTA ? pick<NA>(S.fp, k) : 0.0, fpo = DELTA ? sum_others<NA>(S.fp, k) : 0.0;
        const int r0 = pick<NA>(S.r0, k), r1 = pick<NA>(S.r1, k);
        double o, a;
        if (lg.G == 1) {
            double o4[4] = {0.0, 0.0, 0.0, 0.0}, a4[4] = {0.0, 0.0, 0.0, 0.0};
            int u = r0;
#pragma unroll 1
            for (; u + 4 <= r1; u += 4) {
#pragma unroll
                for (int v = 0; v < 4; ++v) em_bin<MODE>(bins[u + v], lut, ltab, fk, fo, fpk, fpo, o4[v], a4[v], xl[v], bad);
            }
#pragma unroll
            for (int v = 0; v < 3; ++v)
                if (u + v < r1) em_bin<MODE>(bins[u + v], lut, ltab, fk, fo, fpk, fpo, o4[v], a4[v], xl[v], bad);
            o = sum4(o4); a = sum4(a4);
        } else {
            double o1 = 0.0, a1 = 0.0;
#pragma unroll 2
            for (int u = r0 + lg.gl; u < r1; u += 4) em_bin<MODE>(bins[u], lut, ltab, fk, fo, fpk, fpo, o1, a1, xl[0], bad);
            o = lg.sum4(o1); a = lg.sum4(a1);
        }
        put<NA>(o_run, k, o);
        put<NA>(a_run, k, a);
    }
    double x = 0.0;
    if (MODE != kPassPlain) {
        x = lg.G == 1 ? sum4(xl) : lg.sum4(xl[0]);
        if (lg.any(bad != 0u)) x = em_sum_slow<NA, MODE>(bins, S, lut, lg);
    }
    double t_out = 0.0;
    if (S.c_out != 0.0) {
        double F = S.f[0], Fp = S.fp[0];
#pragma unroll
        for (int k = 1; k < NA; ++k) { F += S.f[k]; Fp += S.fp[k]; }
        const double inv = rcp_fast(F);
        t_out = S.c_out * inv;
        if (DELTA) x += S.c_out * fabs(log_ratio(Fp * inv));
    }
#pragma unroll
    for (int k = 0; k < NA; ++k) s[k] = S.f[k] * ((o_run[k] + sum_others<NA>(a_run, k)) + t_out);
    return x;
}

// BV_EM_ABS_INT_TRUNC, the rare case the frequencies cannot decide: is there a bin whose log marginal moved by >= 1?
// ((double)abs((int)diff) is non-zero iff |diff| >= 1; NaN / inf convert to INT_MIN whose "abs" stays negative.)
__device__ __forceinline__ bool moved_by_one(double m, double mp) {
    if (m < 2.5 * mp && mp < 2.5 * m) return false;
    const double diff = nlog(m) - nlog(mp);
    return fabs(diff) >= 1.0 && fabs(diff) < 2147483648.0;
}
template <int NA>
__device__ __noinline__ bool em_moved_bin(const uint32_t* bins, const EmState<NA>& S, const double* lut, const LaneGroup& lg) {
    if (S.c_out != 0.0) {   // the bins outside the subset: marginals e3 * F
        double F = S.f[0], Fp = S.fp[0];
#pragma unroll
        for (int k = 1; k < NA; ++k) { F += S.f[k]; Fp += S.fp[k]; }
        if (moved_by_one(F, Fp)) return true;
    }
    bool found = false;
#pragma unroll 1
    for (int k = 0; k < NA; ++k) {
        const double fk = pick<NA>(S.f, k), fo = sum_others<NA>(S.f, k), fpk = pick<NA>(S.fp, k), fpo = sum_others<NA>(S.fp, k);
        const int r1 = pick<NA>(S.r1, k);
        for (int u = pick<NA>(S.r0, k) + lg.gl; u < r1 && !found; u += lg.G) {   // (a yes / no answer: the order of the visits does not matter)
            const uint32_t q = bin_qual(bins[u]);
            const double ome = lut[kLutOneMinusEps * kQSlots + q], e3 = lut[kLutEpsThird * kQSlots + q];
            found = moved_by_one(ome * fk + e3 * fo, ome * fpk + e3 * fpo);
        }
    }
    return lg.any(found);
}

// first bin of each base (bins are sorted by base) and the number of bins
__device__ __forceinline__ void bin_starts(const EmSiteHdr& H, int (&st)[6]) {
    st[0] = 0; st[1] = (int)(H.base_start[0] & 0xffffu); st[2] = (int)(H.base_start[0] >> 16);
    st[3] = (int)(H.base_start[1] & 0xffffu); st[4] = (int)(H.base_start[1] >> 16); st[5] = (int)H.nb;
}

template <int NA>
__device__ __forceinline__ void em_setup(const EmSiteHdr& H, uint32_t subset, EmState<NA>& S) {
    S.total = (double)H.total;
    int st[6];
    bin_starts(H, st);
    uint32_t left = subset;
    uint32_t c_in = 0;
#pragma unroll
    for (int k = 0; k < NA; ++k) {
        const int jk = __ffs(left) - 1;
        left &= left - 1u;
        int b0 = 0, b1 = 0;
        uint32_t d = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) if (jk == b) { b0 = st[b]; b1 = st[b + 1]; d = H.depth[b]; }
        c_in += d;
        S.r0[k] = b0;
        S.r1[k] = b1;
        // initial frequencies: depth/total for the subset's members, NOT renormalised (src/basetype.cpp:93-103)
        S.f[k] = (double)d / S.total;
        S.fp[k] = S.f[k];
    }
    S.c_out = (double)(H.total - c_in);
}

// The whole EM of one candidate subset (src/algorithm.h:210-255; _f, src/basetype.cpp:105-128).  res: log-likelihood under
// the second-to-last frequencies (what _f() sums), the estimated frequencies, flags.  resume: the iterations were run by
// bv_em_iter_kernel, which left the last two frequency vectors in res.
template <int NA>
__device__ __forceinline__ void em_task(const SiteKernelArgs& a, const double* lut, const double2* ltab, const EmSiteHdr* Hg, const uint32_t* bins,
                                        uint32_t subset, double* res, const LaneGroup& lg) {
    // (the header is read where it is needed, not carried in registers through the EM)
    EmState<NA> S;
    em_setup<NA>(*Hg, subset, S);
    double (&f)[NA] = S.f;
    double (&fp)[NA] = S.fp;
    const double total = S.total;
    double s[NA];
    uint64_t flags = 0;
    double ll = 0.0;
    const bool resume = a.em_resume != 0u;
    if (resume) {
        // the log-likelihood under fp: one pass with the previous frequencies in the place of the current ones
#pragma unroll
        for (int k = 0; k < NA; ++k) { f[k] = res[4 + k]; fp[k] = f[k]; }
        flags = (uint64_t)__double_as_longlong(res[8]);
    }
    bool first = !resume;   // the E-step + M-step in front of EM()'s loop: no convergence test
    int it = a.em_max_iter;
    for (;;) {   // (BV_EM_ABS_INT_TRUNC: with fabs the iterations are bv_em_iter_kernel's, and this function resumes after them)
        bool last = resume;
        if (!resume && !first) {
            // EM()'s convergence test after the E-step under f compares its log marginals with those of the E-step under fp
            // (src/algorithm.h:238-250) -- a function of f and fp alone, so it is evaluated BEFORE the E-step, and the E-step that
            // turns out to be the last also sums the log-likelihood.
            // Every marginal is a non-negative combination of the frequencies, so its ratio between two E-steps lies between
            // the smallest and the largest ratio of the frequencies (e = 2.71828...): all of those inside (1/2.718, 2.718) =>
            // no log marginal moved by 1; all >= 2.7183 or all <= 1/2.7183 => every one did; otherwise the bins decide.
            bool calm = true, up = true, down = true;
#pragma unroll
            for (int k = 0; k < NA; ++k) {
                calm = calm && f[k] < 2.718 * fp[k] && fp[k] < 2.718 * f[k];
                up = up && f[k] >= 2.7183 * fp[k] && fp[k] > 0.0 && f[k] < 1e300;
                down = down && fp[k] >= 2.7183 * f[k] && f[k] > 0.0 && fp[k] < 1e300;
            }
            const bool more = calm ? false : (up || down) ? true : em_moved_bin<NA>(bins, S, lut, lg);
            last = !more || it == 1;
        }
        if (last) ll = em_pass<NA, kPassLL>(bins, S, lut, ltab, s, lg);
        else em_pass<NA, kPassPlain>(bins, S, lut, ltab, s, lg);
        if (resume) {
#pragma unroll
            for (int k = 0; k < NA; ++k) f[k] = res[k];
            break;
        }
#pragma unroll
        for (int k = 0; k < NA; ++k) { fp[k] = f[k]; f[k] = s[k] / total; }
        if (first) { first = false; continue; }
        --it;
        if (it == 0) flags |= BV_FLAG_EM_MAXITER;
        if (last) break;
    }
    // ll: sum of c * log marginal under fp, the frequencies of the last E-step, over the bins of the subset's bases; a bin outside
    // them has the marginal e3(q) * F: log e3 comes from the table, log F is one logarithm for all of them.
    if (S.c_out != 0.0) {
        // the bins outside the subset: table look-ups only, summed in bin order by every lane of the group alike
        int st[6];
        bin_starts(*Hg, st);
        double lo = 0.0;
#pragma unroll 1
        for (int b = 0; b < 5; ++b) {
            if (subset >> b & 1u) continue;
            for (int i = st[b]; i < st[b + 1]; ++i) {
                const uint32_t p = bins[i];
                lo += (double)bin_count(p) * lut[kLutLogMis * kQSlots + bin_qual(p)];
            }
        }
        double F = fp[0];
#pragma unroll
        for (int k = 1; k < NA; ++k) F += fp[k];
        ll += lo + S.c_out * log(F);
    }
    if (lg.gl != 0) return;
    double fo[4] = {0.0, 0.0, 0.0, 0.0};
    uint32_t left = subset;
#pragma unroll
    for (int k = 0; k < NA; ++k) {
        const int jk = __ffs(left) - 1;
        left &= left - 1u;
#pragma unroll
        for (int b = 0; b < 4; ++b) if (jk == b) fo[b] = f[k];
    }
    res[0] = ll; res[1] = fo[0]; res[2] = fo[1]; res[3] = fo[2]; res[4] = fo[3];
    res[5] = __longlong_as_double((long long)flags);
}

// =====================================================================================================================
// bv_em_iter_kernel (BV_EM_ABS_DOUBLE only): the EM iterations, lanes fed task by task.
// With fabs in the convergence test an EM runs anywhere from 5 to 100 iterations, and 32 EMs started together keep their
// warp until the slowest is done.  Here a lane that finishes an EM takes the next task of the list at once (its site's bins
// into the lane's own staging row) and joins the warp's next pass: every pass of the warp carries 32 live EMs, whatever
// iteration each of them is in.  The frequencies of the last two E-steps go to em_res; bv_em_task_kernel then runs the
// (one pass, equal for all) log-likelihood sums and the decisions from there (SiteKernelArgs::em_resume).
// =====================================================================================================================
template <int NA>
__device__ __forceinline__ void em_iter_list(const SiteKernelArgs& a, TaskCta& cs, const double* lut, uint32_t list_base, uint32_t n_list,
                                             uint32_t* fetch) {
    const int lane = threadIdx.x & 31;
    LaneGroup lg;
    lg.G = 1; lg.gl = 0; lg.mask = 1u << lane;
    uint32_t* const my_row = cs.bins + threadIdx.x * kStageStride;
    bool have = false, done = false, first = true;
    uint32_t t = 0;
    int it = 0;
    uint64_t flags = 0;
    const uint32_t* bins = my_row;
    EmState<NA> S;
    S.c_out = 0.0; S.total = 1.0;
#pragma unroll
    for (int k = 0; k < NA; ++k) { S.f[k] = 0.0; S.fp[k] = 0.0; S.r0[k] = 0; S.r1[k] = 0; }
    for (;;) {
        const uint32_t need = __ballot_sync(kFull, !have && !done);
        if (need) {
            uint32_t base = 0;
            if (lane == __ffs(need) - 1) base = atomicAdd(fetch, (uint32_t)__popc(need));
            base = __shfl_sync(kFull, base, __ffs(need) - 1);
            if (!have && !done) {
                const uint32_t idx = base + (uint32_t)__popc(need & ((1u << lane) - 1u));
                if (idx >= n_list) done = true;
                else {
                    t = list_base + idx;
                    const uint32_t word = a.em_tasks[t];
                    const EmSiteHdr H = a.em_hdr[word & 0x0fffffffu];
                    if (H.nb <= (uint32_t)kStageBins) {
                        for (uint32_t i = 0; i < H.nb; ++i) my_row[i] = a.em_pool[H.bins_off + i];
                        bins = my_row;
                    } else bins = a.em_pool + H.bins_off;
                    em_setup<NA>(H, word >> 28, S);
                    have = true; first = true; it = a.em_max_iter; flags = 0;
                }
            }
        }
        if (__ballot_sync(kFull, have) == 0u) {
            if (__ballot_sync(kFull, !done) == 0u) break;
            continue;
        }
        double s[NA];
        const double delta = em_pass<NA, kPassDelta>(bins, S, lut, cs.ltab, s, lg);
        if (have) {
#pragma unroll
            for (int k = 0; k < NA; ++k) { S.fp[k] = S.f[k]; S.f[k] = s[k] / S.total; }
            bool fin = false;
            if (first) first = false;   // the E-step + M-step in front of EM()'s loop: no convergence test
            else {
                --it;
                if (it == 0) flags |= BV_FLAG_EM_MAXITER;
                fin = (delta < a.em_eps) || it == 0;
            }
            if (fin) {
                double* res = a.em_res + (size_t)t * kEmResDoubles;
#pragma unroll
                for (int k = 0; k < NA; ++k) { res[k] = S.f[k]; res[4 + k] = S.fp[k]; }
                res[8] = __longlong_as_double((long long)flags);
                have = false;
                S.c_out = 0.0;
#pragma unroll
                for (int k = 0; k < NA; ++k) { S.r0[k] = 0; S.r1[k] = 0; }
            }
        }
    }
}

__global__ void __launch_bounds__(kTaskThreads) bv_em_iter_kernel(const __grid_constant__ SiteKernelArgs a) {
    TaskCta& cs = *reinterpret_cast<TaskCta*>(bv_smem_raw);
    for (int i = threadIdx.x; i < 4 * kQSlots; i += kTaskThreads) cs.lut[i / kQSlots][i % kQSlots] = a.lut[(i / kQSlots) * kQStride + i % kQSlots];
    for (int i = threadIdx.x; i < kLogTabEntries; i += kTaskThreads) cs.ltab[i] = a.logtab[i];
    __syncthreads();
    grid_dep_wait();
    const double* lut = &cs.lut[0][0];
    em_iter_list<2>(a, cs, lut, 0u, a.counters[kCntEmTask2], a.counters + kCntEmFetch2);
    em_iter_list<3>(a, cs, lut, a.em_task_cap[0], a.counters[kCntEmTask3], a.counters + kCntEmFetch3);
    em_iter_list<4>(a, cs, lut, a.em_task_cap[0] + a.em_task_cap[1], a.counters[kCntEmTask4], a.counters + kCntEmFetch4);
    grid_dep_launch();
}

// ---- the site's decision, after its last task has finished ----------------------------------------------------------------------
// Backward elimination (src/basetype.cpp:144-168) on the task results, ALT / AF / QUAL (:170-196), FS of the VCF row.
// The strand-bias test of a VCF row whose called ALT set is not "every non-reference base" is a Fisher test of its own (ref vs the
// called alleles) -- on a deep pileup a walk of hundreds of steps, needed by one decided site in three.  Run inside the decision it
// kept a few lanes of one or two warps busy while the CTA's other warps waited at the round's barrier (a fifth of this kernel's warp
// time on deep multi-allelic pileups).  The decision only names the test (fs_entry = site | kFisherVcfRow | kFisherWide, 0 = none);
// the caller hands it on to bv_fisher_kernel's list (fisher_push in bv_finish_kernels.cuh).
__device__ __noinline__ void decide_site(const SiteKernelArgs& a, const EmSiteHdr& H, uint32_t hdr_index, uint32_t& fs_entry) {
    const uint32_t site = H.site;
    bv_site_out* rec = a.out + site;
    const int ref_code = ref_code_of(a.ref_base[site]);
    const uint32_t dep[4] = {H.depth[0], H.depth[1], H.depth[2], H.depth[3]};
    const uint32_t total = H.total;
    const double dtot = (double)total;
    const uint32_t act0 = H.act_flags & 0xfu;
    uint32_t act = act0;
    int n_act = __popc(act);
    uint32_t flags = H.act_flags >> 8;
    // result of the task of subset `sub`: tasks of one size are listed in ascending subset order
    auto result = [&](uint32_t sub) {
        const int k = __popc(sub);
        uint32_t below = 0;
        for (uint32_t m = 3; m < sub; ++m) below += ((m & ~act0) == 0u && __popc(m) == k) ? 1u : 0u;
        return a.em_res + (size_t)(H.task[k - 2] + below) * kEmResDoubles;
    };
    const double* r0 = result(act);
    double lr_alt = __ldcg(r0);
    double res_f[4] = {__ldcg(r0 + 1), __ldcg(r0 + 2), __ldcg(r0 + 3), __ldcg(r0 + 4)};
    flags |= (uint32_t)__double_as_longlong(__ldcg(r0 + 5));
    double chi = 0.0;
    uint32_t em_calls = 1;
#pragma unroll 1
    for (int n = n_act - 1; n > 0; --n) {
        // the n-subsets of the n+1 active bases in the lexicographic order of
        // src/external/combinations.h:19-84: the i-th subset drops the (n-i)-th active base
        double single_ll[2] = {0.0, 0.0};
        if (n == 1) {
            // Log-likelihoods of the two single-allele models (EMs whose answer is closed form; NaN when a phred-0 read of that
            // base exists): K4a left them with the header (single_allele_ll4).
            const int b0 = __ffs(act) - 1, b1 = 31 - __clz(act);
            single_ll[0] = __ldcg(a.em_single + (size_t)hdr_index * 4 + b0);
            single_ll[1] = __ldcg(a.em_single + (size_t)hdr_index * 4 + b1);
        }
        double best_chi = 0, best_lr = 0, best_f[4] = {0, 0, 0, 0};
        uint32_t best_set = 0;
#pragma unroll 1
        for (int i = 0; i <= n; ++i) {
            const uint32_t sub = act & ~(1u << nth_active(kOrderACGT, act, n - i));
            double f0sum = 0.0;   // the subset's initial frequencies, summed in A,C,G,T order
#pragma unroll
            for (int b = 0; b < 4; ++b) f0sum += (sub >> b & 1u) ? (double)dep[b] / dtot : 0.0;
            if (f0sum == 0) flags |= BV_FLAG_ZERO_SUBSET;   // the reference throws (basetype.cpp:113)
            double lr, f[4] = {0, 0, 0, 0};
            if (n == 1) {
                const int single = __ffs(sub) - 1;
                lr = single == __ffs(act) - 1 ? single_ll[0] : single_ll[1];
                const double v = (lr != lr) ? lr : 1.0;
#pragma unroll
                for (int b = 0; b < 4; ++b) if (b == single) f[b] = v;
            } else {
                const double* r = result(sub);
                lr = __ldcg(r); f[0] = __ldcg(r + 1); f[1] = __ldcg(r + 2); f[2] = __ldcg(r + 3); f[3] = __ldcg(r + 4);
                flags |= (uint32_t)__double_as_longlong(__ldcg(r + 5));
            }
            if (em_calls < 255) ++em_calls;
            const double c = 2 * (lr_alt - lr);
            // std::min_element keeps the FIRST minimum (algorithm.h:24-27).  Alleles with identical read
            // multisets have equal likelihood; the reference's pick between them hangs on the rounding noise
            // of its read-order sums.  Values that agree to rounding noise are treated as the tie they are:
            // the earlier subset stays and the site is flagged.
            const double tie_tol = 1e-11 * (fabs(lr_alt) + fabs(lr));
            if (i > 0 && fabs(c - best_chi) <= tie_tol) flags |= BV_FLAG_LRT_TIE;
            if (i == 0 || c < best_chi - tie_tol) {
                best_chi = c; best_lr = lr; best_set = sub;
                best_f[0] = f[0]; best_f[1] = f[1]; best_f[2] = f[2]; best_f[3] = f[3];
            }
        }
        lr_alt = best_lr;
        chi = best_chi;
        const double lrt_threshold = a.lrt_threshold;
        if (fabs(chi - lrt_threshold) < 1e-9 * lrt_threshold) flags |= BV_FLAG_NEAR_LRT;
        if (chi < lrt_threshold) {
            act = best_set; n_act = n;
            res_f[0] = best_f[0]; res_f[1] = best_f[1]; res_f[2] = best_f[2]; res_f[3] = best_f[3];
        } else {
            break;
        }
    }

    // ---- ALT / QUAL (src/basetype.cpp:170-196) ----
    const uint32_t ref_bit = ref_code >= 0 ? (1u << ref_code) : 0u;
    const uint32_t alt_set = act & ~ref_bit;
    const int n_alt = __popc(alt_set);
    double qual = 0.0, fs_vcf = 0.0;
    if (n_alt) {
        const int first_act = __ffs(act) - 1;
        const double r = (double)dep[first_act] / dtot;
        if (n_act == 1 && total > 10 && r > 0.5) { qual = 5000.0; flags |= BV_FLAG_MONO_QUAL; }
        else qual = qual_from_chi(chi);
        // strand bias of the VCF row, ref vs the called ALT alleles (src/basetype.cpp:244-295, basetype_caller.cpp:1164)
        int rf, rr, vf, vr, af_, ar;
        strand_tables(rec, ref_code, alt_set, rf, rr, vf, vr, af_, ar);
        if ((vf | vr) != 0 && (rf | rr) != 0) {
            double p;
            if (fisher_margin1(rf, rr, vf, vr, p)) fs_vcf = fs_from_p(p);
            else   // bv_fisher_kernel completes the record (also when the table is that of the CVG row: its FS is not there yet either)
                fs_entry = site | kFisherVcfRow | (fisher_support_wide(rf, rr, vf, vr) ? kFisherWide : 0u);
        }
    }
    // ---- record: ALT alleles in ACGT order of the active set (src/basetype.cpp:172-177) ----
    uint32_t alts = 0;
    int k = 0;
    double af[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        if (alt_set >> b & 1u) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) if (kk == k) af[kk] = res_f[b];
            alts |= (uint32_t)b << (8 * k);
            ++k;
        }
    }
    uint32_t* w = reinterpret_cast<uint32_t*>(rec);
    w[kWState] = kStateDone;
    w[kWAlt] = (uint32_t)n_alt | (alts << 8);                       // n_alt, alt[0..2]
    w[kWInfo] = (alts >> 24) | ((uint32_t)n_act << 8) | ((flags & 0xffu) << 16) | (em_calls << 24);   // alt[3], n_active, flags, em_calls
    rec->af[0] = af[0]; rec->af[1] = af[1]; rec->af[2] = af[2]; rec->af[3] = af[3];
    rec->qual = qual;
    rec->chi2 = chi;
    rec->fs_vcf = fs_vcf;
    // called sites go on to the rank-sum / population-group kernels (bv_call_kernels.cuh)
    if (n_alt && a.list_called) a.list_called[atomicAdd(a.counters + kCntCalled, 1u)] = site;
}

// Two builds of the kernel, launched one after the other; the task count (known on the device only) picks the one that works,
// the other leaves at once.  kMinCtas = kTaskLoCtas (3): 168 registers, three CTAs per SM, fastest while the tasks of a tile
// fit one round of resident threads.  kMinCtas = kTaskHiCtas (4): 128 registers (and 384 bytes of spill stores), four CTAs per
// SM, 12 % faster once they do not (deep multi-allelic pileups: 185,000 tasks per 200,000 sites of C5) and 7-14 % slower below
// (register counts from ptxas -v; timings on a B200 in profiles/r02_em_task_occupancy.txt).
template <int kMinCtas>
__global__ void __launch_bounds__(kTaskThreads, kMinCtas) bv_em_task_kernel(const __grid_constant__ SiteKernelArgs a) {
    TaskCta& cs = *reinterpret_cast<TaskCta*>(bv_smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    for (int i = tid; i < 4 * kQSlots; i += kTaskThreads) cs.lut[i / kQSlots][i % kQSlots] = a.lut[(i / kQSlots) * kQStride + i % kQSlots];
    for (int i = tid; i < kLogTabEntries; i += kTaskThreads) cs.ltab[i] = a.logtab[i];
    if (tid == 0) cs.n_fs = 0;
    grid_dep_wait();
    {
        const uint64_t n_all = (uint64_t)a.counters[kCntEmTask2] + a.counters[kCntEmTask3] + a.counters[kCntEmTask4];
        if ((n_all > (uint64_t)a.em_task_split) != (kMinCtas == kTaskHiCtas)) return;
    }
    const double* lut = &cs.lut[0][0];
    // the three task lists, one after the other
    uint32_t n_list[3], blk_end[3], base[3];
    n_list[0] = a.counters[kCntEmTask2];
    n_list[1] = a.counters[kCntEmTask3];
    n_list[2] = a.counters[kCntEmTask4];
    base[0] = 0; base[1] = a.em_task_cap[0]; base[2] = a.em_task_cap[0] + a.em_task_cap[1];
    // Lanes per task: one -- a thread per task -- unless the tile has so few tasks that most of the GPU would stand idle
    // behind their serial chains: then four (the sums are formed the same way either way, see LaneGroup).
    LaneGroup lg;
    {
        const uint64_t n_tasks = (uint64_t)n_list[0] + n_list[1] + n_list[2];
        const int G = n_tasks <= (uint64_t)kG4MaxTasks ? 4 : 1;
        lg.G = G;
        lg.gl = lane & (G - 1);
        lg.mask = (G == 1 ? 1u : 0xfu) << (lane & ~(G - 1));
    }
    const uint32_t tpc = (uint32_t)(kTaskThreads / lg.G);   // tasks per CTA and round
    const uint32_t slot = (uint32_t)tid / (uint32_t)lg.G;    // this thread's task of the round = its staging row
    blk_end[0] = (n_list[0] + tpc - 1) / tpc;
    blk_end[1] = blk_end[0] + (n_list[1] + tpc - 1) / tpc;
    blk_end[2] = blk_end[1] + (n_list[2] + tpc - 1) / tpc;
#pragma unroll 1
    for (uint32_t v = blockIdx.x; v < blk_end[2]; v += gridDim.x) {
        const int li = v < blk_end[0] ? 0 : v < blk_end[1] ? 1 : 2;   // (CTA-uniform) tasks of one subset size per round
        const uint32_t idx = (v - (li ? blk_end[li - 1] : 0u)) * tpc + slot;
        const uint32_t t = base[li] + idx;
        const uint32_t word = idx < n_list[li] ? a.em_tasks[t] : kEmTaskInvalid;
        const bool valid = word != kEmTaskInvalid;
        const uint32_t hdr = word & 0x0fffffffu, subset = word >> 28;
        __syncthreads();   // the previous round's readers of cs.bins are done (first round: the tables are written)
        if (cs.n_fs >= (uint32_t)kTaskThreads) {   // (CTA-uniform) a whole CTA of listed Fisher tests: on to bv_fisher_kernel's list
            const uint32_t e = cs.fs_site[cs.n_fs - (uint32_t)kTaskThreads + (uint32_t)tid];
            fisher_push(a, true, (e & kFisherWide) != 0u, e & ~kFisherWide);
            __syncthreads();
            if (tid == 0) cs.n_fs -= (uint32_t)kTaskThreads;
        }
        if (tid == 0) cs.n_decide = 0;
        EmSiteHdr* const Hg = a.em_hdr + hdr;
        uint32_t h_nb = 0, h_off = 0;   // (only these two words of the header are needed here)
        if (valid) { h_off = Hg->bins_off; h_nb = Hg->nb; }
        // Staging, warp by warp: the tasks of a site are neighbours in the list, so one row serves a run of lanes with the same
        // header; all 32 lanes copy it (coalesced), one run after the other.  Lists longer than a row are read from the pool.
        const uint32_t hdr_prev = __shfl_up_sync(kFull, valid ? hdr : kEmTaskInvalid, 1);
        const bool leader = valid && (lane == 0 || hdr_prev != hdr);
        const uint32_t lead = __ballot_sync(kFull, leader);
        const uint32_t row = (uint32_t)(tid & ~31) + (uint32_t)__popc(lead & ((2u << lane) - 1u)) - 1u;   // row of the last leader up to this lane
        for (uint32_t todo = lead; todo; todo &= todo - 1u) {
            const int src = __ffs(todo) - 1;
            const uint32_t nb = __shfl_sync(kFull, h_nb, src), off = __shfl_sync(kFull, h_off, src);
            const uint32_t r = (uint32_t)(tid & ~31) + (uint32_t)__popc(lead & ((2u << src) - 1u)) - 1u;
            if (nb <= (uint32_t)kStageBins)
                for (uint32_t i = lane; i < nb; i += 32) cs.bins[r * kStageStride + i] = a.em_pool[off + i];
        }
        const uint32_t* bins = nullptr;
        if (valid) bins = h_nb <= (uint32_t)kStageBins ? cs.bins + row * kStageStride : a.em_pool + h_off;
        __syncthreads();
        if (valid) {
            double* res = a.em_res + (size_t)t * kEmResDoubles;
            if (li == 0) em_task<2>(a, lut, cs.ltab, Hg, bins, subset, res, lg);
            else if (li == 1) em_task<3>(a, lut, cs.ltab, Hg, bins, subset, res, lg);
            else em_task<4>(a, lut, cs.ltab, Hg, bins, subset, res, lg);
            if (lg.gl == 0) {
                __threadfence();
                if (atomicSub(&Hg->remaining, 1u) == 1u) {   // every task of the site has stored its result: queue the decision
                    cs.decide_hdr[atomicAdd(&cs.n_decide, 1u)] = hdr;
                }
            }
        }
        __syncthreads();
        // the decisions of this round, one thread per site (scalar work: a lane per site keeps the warps full)
        if ((uint32_t)tid < cs.n_decide) {
            __threadfence();
            const EmSiteHdr Hd = a.em_hdr[cs.decide_hdr[tid]];
            uint32_t e = 0;
            decide_site(a, Hd, cs.decide_hdr[tid], e);
            if (e) cs.fs_site[atomicAdd(&cs.n_fs, 1u)] = e;
        }
    }
    __syncthreads();
    grid_dep_launch();
    for (uint32_t k0 = 0; k0 < cs.n_fs; k0 += (uint32_t)kTaskThreads) {   // the tests still listed here
        const bool have = k0 + (uint32_t)tid < cs.n_fs;
        const uint32_t e = have ? cs.fs_site[k0 + (uint32_t)tid] : 0u;
        fisher_push(a, have, (e & kFisherWide) != 0u, e & ~kFisherWide);
    }
}

}  // namespace bv
