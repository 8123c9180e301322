// bv_finish_kernels.cuh -- K2 (scalar finish, one thread per site), K3 (likelihood-ratio bound, one warp per site) and the
// warp-per-site device code (row histogram, EM on bins, LRT) that K4a (bv_em_kernels.cuh) and K6 (bv_call_kernels.cuh) share.
// See bv_common.cuh for the split of the basetype core into kernels.
#pragma once
#include "bv_common.cuh"
#include "bv_math.cuh"

namespace bv {

// =====================================================================================================================
// K2: one thread per site of K1's work list (the row has reads that differ from REF, or REF is not A/C/G/T, or a
// bad strand code).  Everything here is a function of the nine counts K1 left in the record:
//   * active alleles: depth/total >= min_af                                            (src/basetype.cpp:135-139)
//   * strand bias of the CVG row, ref vs all non-ref ACGT: two-sided Fisher, FS         (src/basetype.cpp:244-295,
//                                                                                        basetype_caller.cpp:1236-1245)
// If exactly one allele is active and it is REF the record is final (the reference's single-column EM gives f = 1, no
// ALT).  Otherwise the result depends on base qualities: state kStateBound when the site has the shape the bound of K3
// can decide (REF with >= 22 reads plus one minor allele with <= 4, and lrt_threshold >= 24; the minor allele's code travels
// in the alt word), else state kStateEM.
// =====================================================================================================================
// append `site` to a work list (global, or a CTA's staging list in shared memory) for the lanes with `pred`; one atomicAdd
// per warp (all 32 lanes must call)
__device__ __forceinline__ void list_append(uint32_t* list, uint32_t* counter, bool pred, uint32_t site) {
    const int lane = threadIdx.x & 31;
    const uint32_t m = __ballot_sync(kFull, pred);
    if (m == 0) return;
    uint32_t pos = 0;
    if (lane == __ffs(m) - 1) pos = atomicAdd(counter, (uint32_t)__popc(m));
    pos = __shfl_sync(kFull, pos, __ffs(m) - 1);
    if (pred) list[pos + __popc(m & ((1u << lane) - 1u))] = site;
}

// Fisher tests that are not closed form are not run where they arise.  A test is a walk over the table's support: <= 24 outcomes
// the reference's own way (kt_fisher_exact), or bisection + tail sums for wider supports (bv_fisher_fast.h) -- two paths that share
// no code and cost 10-100x the rest of a site.  Run lane by lane, each lane on its own site, a warp executed both paths for every
// mixed group of 32 sites (8 of 32 lanes active on deep pileups), and queues per CTA left most warps waiting for the CTA's few wide
// tests (41 % of K2's warp time at a barrier, profiles/r02_fisher_queues.txt).  So K2 (the CVG row's test) and the decisions of K4b
// (the VCF row's) only LIST their tests, by support width, and bv_fisher_kernel runs them all after K4b: every warp on one path,
// the whole GPU on the wide ones first.
// all 32 lanes call; `entry` of the lanes with pred goes onto the narrow or the wide end of list_fisher
__device__ __forceinline__ void fisher_push(const SiteKernelArgs& a, bool pred, bool wide, uint32_t entry) {
    const int lane = threadIdx.x & 31;
    const uint32_t below = (1u << lane) - 1u;
    const uint32_t mn = __ballot_sync(kFull, pred && !wide), mw = __ballot_sync(kFull, pred && wide);
    if (mn) {
        uint32_t pos = 0;
        if (lane == __ffs(mn) - 1) pos = atomicAdd(a.counters + kCntFisherNarrow, (uint32_t)__popc(mn));
        pos = __shfl_sync(kFull, pos, __ffs(mn) - 1);
        if (pred && !wide) a.list_fisher[pos + __popc(mn & below)] = entry;
    }
    if (mw) {
        uint32_t pos = 0;
        if (lane == __ffs(mw) - 1) pos = atomicAdd(a.counters + kCntFisherWide, (uint32_t)__popc(mw));
        pos = __shfl_sync(kFull, pos, __ffs(mw) - 1);
        if (pred && wide) a.list_fisher[2u * a.n_sites - 1u - (pos + __popc(mw & below))] = entry;
    }
}
// Which end of the list: is the support [max(0, n1_ + n_1 - n), min(n1_, n_1)] of the table (a b / c d) wider than kFisherListWide
// outcomes?  24 = where the algorithm changes (fisher_fast_applicable): the reference's walk on one end, bisection + tails on the
// other.  Splitting later (48, 96, 200: the cheap bisections with the walks, only the long tails apart) measured slower on deep pileups
// (bv_fisher_kernel on C5: 0.256 / 0.279 / 0.315 / 0.342 ms per 10^6 sites), equal elsewhere (profiles/r02_fisher_queues.txt).
constexpr int kFisherListWide = 24;
__device__ __forceinline__ bool fisher_support_wide(int t11, int t12, int t21, int t22) {
    const int n1_ = t11 + t12, n_1 = t11 + t21, n = n1_ + t21 + t22;
    return min(n1_, n_1) - max(0, n1_ + n_1 - n) > kFisherListWide;
}

// The two strand tables of a site from its record: ref vs every non-reference base (CVG row, basetype_caller.cpp:1236-1245) and ref
// vs the called ALT alleles (VCF row, :1164); src/basetype.cpp:244-295.
__device__ __forceinline__ void strand_tables(const bv_site_out* rec, int ref_code, uint32_t alt_set, int& rf, int& rr, int& vf, int& vr,
                                              int& af_, int& ar) {
    const uint32_t f[4] = {rec->fwd[0], rec->fwd[1], rec->fwd[2], rec->fwd[3]};
    const uint32_t rv[4] = {rec->rev[0], rec->rev[1], rec->rev[2], rec->rev[3]};
    rf = 0; rr = 0; vf = 0; vr = 0; af_ = 0; ar = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        if (b == ref_code) { rf = (int)f[b]; rr = (int)rv[b]; }
        else { af_ += (int)f[b]; ar += (int)rv[b]; }
        if (alt_set >> b & 1u) { vf += (int)f[b]; vr += (int)rv[b]; }
    }
}

// One queued test (all 32 lanes call): the table again from the site's (by now final) record, the test, FS into the record.
// pair: lanes 2k and 2k + 1 share the test, the even lane sums its left tail, the odd one its right tail -- half the latency of the
// kernel's longest dependency chain, which is all that counts while the tests of a tile leave most of the GPU's threads unused.
// left + right is the very sum the one-thread test forms, so the value is the same bit for bit in both modes (and in bv_fs_kernel).
__device__ __forceinline__ void fisher_job(const SiteKernelArgs& a, bool have, uint32_t entry, bool pair) {
    const int side = pair ? (int)(threadIdx.x & 1u) : kFisherBoth;
    double part = 0.0;
    bool whole = false;
    bv_site_out* rec = nullptr;
    if (have) {
        const uint32_t site = entry & 0x00ffffffu;
        rec = a.out + site;
        const int ref_code = ref_code_of(a.ref_base[site]);
        uint32_t alt_set = 0;
        if (entry & kFisherVcfRow)
            for (int k = 0; k < (int)rec->n_alt; ++k) alt_set |= 1u << (rec->alt[k] & 3u);
        int rf, rr, vf, vr, af_, ar;
        strand_tables(rec, ref_code, alt_set, rf, rr, vf, vr, af_, ar);
        if (!(entry & kFisherVcfRow)) { vf = af_; vr = ar; }
        part = fisher_two_sided(a.logfact, rf, rr, vf, vr, side, &whole);   // (margin-1 tables are closed form and never listed)
    }
    const double other = __shfl_xor_sync(kFull, part, 1);
    if (have && side != kFisherRight) {
        double p = (pair && !whole) ? part + other : part;
        if (p > 1.) p = 1.;
        const double fs = fs_from_p(p);
        if (entry & kFisherVcfRow) rec->fs_vcf = fs; else rec->fs_cvg = fs;
    }
}

constexpr int kFisherThreads = 256;
__global__ void __launch_bounds__(kFisherThreads) bv_fisher_kernel(const __grid_constant__ SiteKernelArgs a) {
    grid_dep_wait();
    const uint32_t n_wide = a.counters[kCntFisherWide], n_narrow = a.counters[kCntFisherNarrow];
    const uint32_t threads = gridDim.x * blockDim.x;
    const bool pair = 2u * (n_wide + n_narrow + 32u) <= threads;      // a pair of lanes per test while that still is one trip
    const uint32_t per_warp = pair ? 16u : 32u, shift = pair ? 1u : 0u;
    const uint32_t first_narrow = (n_wide + per_warp - 1u) & ~(per_warp - 1u), n_jobs = first_narrow + n_narrow;   // the narrow tests
                                                                                                       // start on a warp of their own
    for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> shift; (j & ~(per_warp - 1u)) < n_jobs; j += threads >> shift) {   // warp-uniform trips
        bool have = false;
        uint32_t entry = 0;
        if (j < first_narrow) {
            if (j < n_wide) { have = true; entry = a.list_fisher[2u * a.n_sites - 1u - j]; }
        } else if (j < n_jobs) { have = true; entry = a.list_fisher[j - first_narrow]; }
        fisher_job(a, have, entry, pair);
    }
}

// K2 works in passes of kScalarSites sites per thread: the list entries of a pass, then the records and REF bases of all
// of its sites are loaded before the first site is finished, so that a thread has kScalarSites scattered 64-byte reads in
// flight instead of one.  Its appends to the four work lists (bound, EM, narrow and wide Fisher tests) are gathered in
// shared memory and go out with one global atomicAdd per list and CTA: per warp they were four returning atomics in a row
// on four counters that every warp of the tile hit.
constexpr int kScalarThreads = 256;
constexpr int kScalarSites = 4;
constexpr uint32_t kScalarPass = (uint32_t)kScalarThreads * kScalarSites;   // sites per CTA and pass

__device__ __forceinline__ uint32_t scalar_site(const SiteKernelArgs& a, uint32_t site, const uint4 (&w)[4], uint32_t ref_char,
                                                bool& fs_job, bool& fs_wide);

__global__ void __launch_bounds__(kScalarThreads) bv_scalar_kernel(const __grid_constant__ SiteKernelArgs a) {
    __shared__ uint32_t s_list[4][kScalarPass];   // staged appends: bound, EM, narrow Fisher, wide Fisher
    __shared__ uint32_t s_cnt[4], s_n[4], s_base[4];
    const int tid = threadIdx.x;
    if (tid < 4) s_cnt[tid] = 0;
    // every CTA takes an equal slice of the list (all SMs get work however few sites are listed), in passes
    const uint32_t n_slow = a.counters[kCntSlow];
    const uint32_t slice = ((n_slow + gridDim.x - 1u) / gridDim.x + 31u) & ~31u;
    const uint32_t end = min(n_slow, (blockIdx.x + 1u) * slice);
#pragma unroll 1
    for (uint32_t p0 = blockIdx.x * slice; p0 < end; p0 += kScalarPass) {   // CTA-uniform trips
        uint32_t site[kScalarSites], ref_char[kScalarSites];
        uint4 w[kScalarSites][4];
#pragma unroll
        for (int k = 0; k < kScalarSites; ++k) {
            const uint32_t i = p0 + (uint32_t)(k * kScalarThreads + tid);
            site[k] = i < end ? a.list_slow[i] : 0xffffffffu;
        }
#pragma unroll
        for (int k = 0; k < kScalarSites; ++k) {
            if (site[k] != 0xffffffffu) {
                const uint4* rec = reinterpret_cast<const uint4*>(a.out + site[k]);
                w[k][0] = rec[0]; w[k][1] = rec[1]; w[k][2] = rec[2]; w[k][3] = rec[3];
                ref_char[k] = a.ref_base[site[k]];
            }
        }
        __syncthreads();   // s_cnt is zero and the previous pass's staging lists are written out
#pragma unroll
        for (int k = 0; k < kScalarSites; ++k) {
            const bool valid = site[k] != 0xffffffffu;
            bool fs_job = false, fs_wide = false;
            const uint32_t state = valid ? scalar_site(a, site[k], w[k], ref_char[k], fs_job, fs_wide) : kStateDone;
            list_append(s_list[0], &s_cnt[0], state == kStateBound, site[k]);
            list_append(s_list[1], &s_cnt[1], state == kStateEM, site[k]);
            list_append(s_list[2], &s_cnt[2], fs_job && !fs_wide, site[k]);
            list_append(s_list[3], &s_cnt[3], fs_job && fs_wide, site[k]);
        }
        __syncthreads();
        if (tid < 4) {
            const int cnt = tid == 0 ? kCntBound : tid == 1 ? kCntEm : tid == 2 ? kCntFisherNarrow : kCntFisherWide;
            const uint32_t n = s_cnt[tid];
            s_n[tid] = n;
            s_base[tid] = n ? atomicAdd(a.counters + cnt, n) : 0u;
            s_cnt[tid] = 0;
        }
        __syncthreads();
        for (uint32_t j = tid; j < s_n[0]; j += kScalarThreads) a.list_bound[s_base[0] + j] = s_list[0][j];
        for (uint32_t j = tid; j < s_n[1]; j += kScalarThreads) a.list_em[s_base[1] + j] = s_list[1][j];
        // narrow tests from the front of list_fisher, wide ones from the back (bv_fisher_kernel)
        for (uint32_t j = tid; j < s_n[2]; j += kScalarThreads) a.list_fisher[s_base[2] + j] = s_list[2][j];
        for (uint32_t j = tid; j < s_n[3]; j += kScalarThreads) a.list_fisher[2u * a.n_sites - 1u - (s_base[3] + j)] = s_list[3][j];
    }
    grid_dep_launch();
}

// returns the site's new state
// w: the first 64 bytes of the site's record, ref_char: its REF base
__device__ __forceinline__ uint32_t scalar_site(const SiteKernelArgs& a, uint32_t site, const uint4 (&w)[4], uint32_t ref_char,
                                                bool& fs_job, bool& fs_wide) {
    uint32_t* rec = reinterpret_cast<uint32_t*>(a.out + site);
    const uint4 w0 = w[0];   // depth[4]
    const uint4 w1 = w[1];   // other, state, fwd[0..1]
    const uint4 w2 = w[2];   // fwd[2..3], rev[0..1]
    const uint4 w3 = w[3];   // rev[2..3], alt word, info word
    const uint32_t d0 = w0.x, d1 = w0.y, d2 = w0.z, d3 = w0.w, other = w1.x;
    const uint32_t f0 = w1.z, f1 = w1.w, f2 = w2.x, f3 = w2.y, r0 = w2.z, r1 = w2.w, r2 = w3.x, r3 = w3.y;
    const uint32_t flags = (w3.w >> 16) & 0xffu;
    const int ref_code = ref_code_of(ref_char);
    const uint32_t total = d0 + d1 + d2 + d3 + other;
    const double dtot = (double)total;

    uint32_t act = 0;
    if (total > 0) {
        act |= is_active(d0, total, dtot, a.min_af) ? 1u : 0u;
        act |= is_active(d1, total, dtot, a.min_af) ? 2u : 0u;
        act |= is_active(d2, total, dtot, a.min_af) ? 4u : 0u;
        act |= is_active(d3, total, dtot, a.min_af) ? 8u : 0u;
    }
    const uint32_t n_act = __popc(act);
    const uint32_t ref_bit = ref_code >= 0 ? (1u << ref_code) : 0u;
    const bool need_qual = n_act >= 2 || (n_act == 1 && (act & ~ref_bit));

    double fs_cvg = 0.0;
    {
        const int rf = ref_code < 0 ? 0 : (int)sel4u(ref_code, f0, f1, f2, f3);
        const int rr = ref_code < 0 ? 0 : (int)sel4u(ref_code, r0, r1, r2, r3);
        const int af_ = (int)(f0 + f1 + f2 + f3) - rf, ar = (int)(r0 + r1 + r2 + r3) - rr;
        // a table with an empty row or column has a single possible outcome: p == 1, FS == 0 (kfunc.c:256)
        if ((af_ | ar) != 0 && (rf | rr) != 0) {
            double p;
            if (fisher_margin1(rf, rr, af_, ar, p)) fs_cvg = fs_from_p(p);
            else { fs_job = true; fs_wide = fisher_support_wide(rf, rr, af_, ar); }   // bv_fisher_kernel completes the record
        }
    }
    uint32_t state = need_qual ? kStateEM : kStateDone;
    // the active set travels in bits 8-11 of the alt word (K4a), the minor allele of a bound site in bits 0-1 (K3)
    if (need_qual) rec[kWAlt] = act << 8;
    // K3's proof ends in 2G < 23.9 < 24 <= lrt_threshold: below 24 its sites are the EM's
    if (n_act == 2 && (act & ref_bit) && a.lrt_threshold >= 24.0) {
        const int o_code = __ffs(act & ~ref_bit) - 1;
        if (sel4u(ref_code, d0, d1, d2, d3) >= 22 && sel4u(o_code, d0, d1, d2, d3) <= 4) {
            state = kStateBound;
            rec[kWAlt] = (uint32_t)o_code | (act << 8);
        }
    }
    // n_active | flags | em_calls (a single active allele costs the reference one EM call)
    const uint32_t em_calls = (!need_qual && n_act == 1) ? 1u : 0u;
    const uint32_t em_flags = em_calls ? single_em_flag(sel4u(__ffs(act) - 1, d0, d1, d2, d3), total, a) : 0u;
    rec[kWInfo] = (n_act << 8) | ((flags | em_flags) << 16) | (em_calls << 24);
    reinterpret_cast<double*>(rec)[14] = fs_cvg;
    rec[kWState] = state;
    return state;
}

// FS of free-standing 2x2 strand tables (bv_fisher_fs): one thread per table, the rule of scalar_site above.
__global__ void __launch_bounds__(128) bv_fs_kernel(const int4* __restrict__ tables, double* __restrict__ fs, uint32_t n,
                                                    const double* __restrict__ logfact) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int4 t = tables[i];   // ref_fwd, ref_rev, alt_fwd, alt_rev
    double v = 0.0;
    if ((t.z | t.w) != 0 && (t.x | t.y) != 0) v = fs_from_table(logfact, t.x, t.y, t.z, t.w);
    fs[i] = v;
}

// =====================================================================================================================
// K7 bv_pack_kernel (BV_OUT_COMPACT tiles, after everything else): the sites K1 could not finish from their counts get their
// full record copied into the list at a.full_out -- for a host tile the slot's mapped pinned staging, which the kernel writes across
// PCIe itself; for a device-resident tile the caller's device buffer -- 8 lanes per 128-byte record, the records of a warp's sites
// next to each other, and their brief becomes the record's index in that list.
// =====================================================================================================================
__global__ void __launch_bounds__(256) bv_pack_kernel(const __grid_constant__ SiteKernelArgs a) {
    const int lane = threadIdx.x & 31;
    const uint32_t n_sites = a.n_sites;
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint4* const src = reinterpret_cast<const uint4*>(a.out);
    uint4* const dst = reinterpret_cast<uint4*>(a.full_out);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; (i & ~31u) < n_sites; i += stride) {   // warp-uniform trips
        const bool need = i < n_sites && a.brief[i].x == 0xffffffffu;
        const uint32_t m = __ballot_sync(kFull, need);
        if (m == 0) continue;
        uint32_t pos = 0;
        if (lane == __ffs(m) - 1) pos = atomicAdd(a.counters + kCntFull, (uint32_t)__popc(m));
        pos = __shfl_sync(kFull, pos, __ffs(m) - 1);
        const uint32_t my_pos = pos + (uint32_t)__popc(m & ((1u << lane) - 1u));
        if (need) a.brief[i] = make_uint2(0x80000000u | my_pos, 0u);
        // four records per step: lanes 8r .. 8r + 7 copy the r-th of them, 16 bytes each
        const uint32_t cnt = (uint32_t)__popc(m);
        for (uint32_t k0 = 0; k0 < cnt; k0 += 4) {
            const uint32_t k = k0 + (uint32_t)(lane >> 3);
            // the k-th set bit of m
            uint32_t mm = m;
            for (uint32_t t = 0; t < k && mm; ++t) mm &= mm - 1u;
            const bool on = k < cnt;
            const int src_lane = on ? __ffs(mm) - 1 : 0;
            const uint32_t site = (i & ~31u) + (uint32_t)src_lane;
            if (on) dst[(size_t)(pos + k) * 8 + (lane & 7)] = src[(size_t)site * 8 + (lane & 7)];
        }
    }
}

// =====================================================================================================================
// K3: one warp per site of the bound list -- a bound that decides the LRT without running the EM.
//
// Site with exactly two active alleles, REF (r) and one other base (o) carried by a few reads: the signature of
// sequencing errors.  With L_ij the per-read likelihoods (src/basetype.cpp:61-64) and g_i = log(1-eps_i) - log(eps_i/3):
//   * every log-likelihood the EM can report for {r,o} is a sum of log(sum_j L_ij f_j) with sum_j f_j <= 1, hence
//       LL{r,o} <= sum_i log(max_j L_ij) = LL{r} + sum_{reads of o} g_i        (all phred >= 2, so 1-eps > eps/3)
//     where LL{r} = sum_{reads of r} log(1-eps_i) + sum_{other reads} log(eps_i/3) is the closed form of the
//     single-allele model (see single_allele_ll);
//   * LL{r} - LL{o} = sum_{reads of r} g_i - sum_{reads of o} g_i >= 0.56 * depth[r] - G,  G = sum_{reads of o} g_i.
// So when 2G < 23.9 and depth[r] >= 22, the first LRT round (src/basetype.cpp:151-168) picks subset {r}
// (chi_r < chi_o) with chi_r = 2 (LL{r,o} - LL{r}) <= 2G < 24 = LRT_THRESHOLD and drops o: the site ends with the
// single active allele REF, no ALT, whatever the EM would have returned.  Margins (23.9 vs 24, G rounded up in fixed
// point) dwarf the 1e-12 rounding noise of the reference's sums.  A counted read with phred < 2 or > 93 voids the
// argument; such a site goes to the EM kernel like the ones whose G is too large.
// The last step, 23.9 < 24 <= lrt_threshold, needs lrt_threshold >= 24: below that K2 lists no site here and the EM decides
// them all (a limit derived from the threshold would have to re-prove the depth[r] >= 22 condition for every threshold).
//
// Light kernel, high occupancy: the row's base + qual planes come through two TMA-filled buffers per warp, the next
// unit (also the next site's first one) in flight while the current one is scanned with SIMD byte arithmetic.
// =====================================================================================================================
constexpr int kBoundWarps = 32;
constexpr int kBChunk = 1024;                 // cells per buffer and plane: two 16-cell vectors per lane
constexpr uint32_t kBoundLimit = 12530483u;   // floor(11.95 * 2^20)

struct __align__(128) BoundBuf {
    uint8_t base[kBChunk];
    uint8_t qual[kBChunk];
};
struct __align__(128) BoundWarp {
    BoundBuf buf[2];
    uint64_t bar[2];
};
struct __align__(128) BoundCta {
    uint32_t gfix[kQSlots];      // ceil(2^20 * (log(1-eps(q)) - log(eps(q)/3))) + 1: g in fixed point, rounded up
};
constexpr size_t kBoundSmemBytes = sizeof(BoundCta) + (size_t)kBoundWarps * sizeof(BoundWarp);
static_assert(kBoundSmemBytes <= 232448, "shared memory of the bound kernel exceeds 227 KB");

__global__ void __launch_bounds__(kBoundWarps * 32, 1) bv_bound_kernel(const __grid_constant__ SiteKernelArgs a) {
    BoundCta& cs = *reinterpret_cast<BoundCta*>(bv_smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    BoundWarp& W = reinterpret_cast<BoundWarp*>(bv_smem_raw + sizeof(BoundCta))[warp];
    for (int q = threadIdx.x; q < kQSlots; q += blockDim.x) {
        const double g = a.lut[kLutLogMatch * kQStride + q] - a.lut[kLutLogMis * kQStride + q];
        cs.gfix[q] = (q >= 2 && q <= BV_QUAL_MAX) ? (uint32_t)ceil(g * 1048576.0) + 1u : 0x01000000u;
    }
    if (lane == 0) {
        mbar_init(&W.bar[0], 1);
        mbar_init(&W.bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    grid_dep_wait();   // (the prologue above reads constant inputs only)

    const uint32_t N = a.n_samples;
    const uint32_t row_bytes = (N + 15u) & ~15u;
    const uint64_t pitch = a.pitch;
    const uint32_t total_warps = gridDim.x * kBoundWarps;
    const uint32_t n_bound = a.counters[kCntBound];
    const uint32_t n_groups = (n_bound + 31u) >> 5;
    uint32_t* const g_out = reinterpret_cast<uint32_t*>(a.out);
    const uint32_t s_buf0 = smem_u32(&W.buf[0]), s_bar0 = smem_u32(&W.bar[0]);
    uint32_t p_buf = 0, c_buf = 0, phase = 0;   // buffers alternate over the whole unit stream of this warp

#pragma unroll 1
    for (uint32_t g = blockIdx.x * kBoundWarps + warp; g < n_groups; g += total_warps) {
        // 32 consecutive entries of the work list: lane l looks after entry l, the warp scans them one after the other
        const bool valid = g * 32u + lane < n_bound;
        const uint32_t my_site = valid ? a.list_bound[g * 32u + lane] : 0u;
        const uint32_t todo = __ballot_sync(kFull, valid);
        uint32_t my_o = 0, my_info = 0, my_act = 0;
        if (valid) {
            my_o = g_out[(size_t)my_site * 32 + kWAlt];
            my_act = my_o & 0xf00u;
            my_o &= 3u;
            my_info = g_out[(size_t)my_site * 32 + kWInfo];
        }
        // producer cursor over the units (site, chunk) of this group: one unit ahead of the scan
        uint32_t p_todo = todo, p_off = 0;
        uint32_t p_site = __shfl_sync(kFull, my_site, __ffs(p_todo) - 1);
        p_todo &= p_todo - 1u;
        bool p_valid = true;
        auto issue = [&]() {
            if (p_valid) {
                if (lane == 0) {
                    const uint32_t bytes = min((uint32_t)kBChunk, row_bytes - p_off);
                    const uint32_t bar = s_bar0 + 8u * p_buf, dst = s_buf0 + (uint32_t)sizeof(BoundBuf) * p_buf;
                    mbar_expect_tx(bar, 2u * bytes);
                    bulk_g2s(dst, a.base + (size_t)p_site * pitch + p_off, bytes, bar);
                    bulk_g2s(dst + (uint32_t)kBChunk, a.qual + (size_t)p_site * a.qual_pitch + p_off, bytes, bar);
                }
                p_buf ^= 1u;
                p_off += kBChunk;
                if (p_off >= row_bytes) {
                    p_off = 0;
                    // (warp-uniform branch: every lane takes part in the shuffle)
                    if (p_todo) { p_site = __shfl_sync(kFull, my_site, __ffs(p_todo) - 1); p_todo &= p_todo - 1u; }
                    else p_valid = false;
                }
            }
        };
        issue();
        uint32_t c_todo = todo;
#pragma unroll 1
        while (c_todo) {
            const int l = __ffs(c_todo) - 1;
            c_todo &= c_todo - 1u;
            const uint32_t ow = __shfl_sync(kFull, my_o, l) * 0x01010101u;
            uint32_t G = 0, bad = 0;
#pragma unroll 1
            for (uint32_t c_off = 0; c_off < row_bytes; c_off += kBChunk) {
                issue();   // goes into the buffer the previous unit used; every lane is past it (__syncwarp below)
                mbar_wait(s_bar0 + 8u * c_buf, (phase >> c_buf) & 1u);
                phase ^= 1u << c_buf;
#pragma unroll
                for (int v = 0; v < kBChunk / 512; ++v) {
                    const int lane_cells = (int)N - (int)c_off - v * 512 - lane * 16;
                    if (lane_cells > 0) {
                        const uint8_t* cellp = W.buf[c_buf].base + v * 512 + lane * 16;
                        uint4 vb = *reinterpret_cast<const uint4*>(cellp);
                        const uint4 vq = *reinterpret_cast<const uint4*>(cellp + kBChunk);
                        if (lane_cells < 16) mask_tail(vb, lane_cells);
                        const uint32_t wb[4] = {vb.x, vb.y, vb.z, vb.w}, wq[4] = {vq.x, vq.y, vq.z, vq.w};
                        uint32_t eo[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const uint32_t m = ~(((wb[k] | 0x80808080u) - 0x05050505u) | wb[k]) & 0x80808080u;   // counted
                            const uint32_t q7 = wq[k] & 0x7f7f7f7fu;
                            bad |= (~(q7 + 0x7e7e7e7eu) | (q7 + 0x22222222u) | wq[k]) & m;                        // phred < 2 or > 93
                            const uint32_t x = (wb[k] ^ ow) & 0x7f7f7f7fu;
                            eo[k] = ~((x + 0x7f7f7f7fu) | wb[k]) & 0x80808080u;                                   // base == o
                        }
                        if (eo[0] | eo[1] | eo[2] | eo[3]) {
                            uint32_t t = (eo[0] >> 7) | (eo[1] >> 6) | (eo[2] >> 5) | (eo[3] >> 4);   // bit (8*byte + word)
                            do {
                                int top;
                                asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(t));
                                t ^= 1u << top;
                                const int cell = ((top & 3) << 2) | (top >> 3);
                                const uint32_t q = cellp[cell + kBChunk];
                                G += cs.gfix[min(q, (uint32_t)(kQSlots - 1))];
                            } while (t);
                        }
                    }
                }
                __syncwarp();
                c_buf ^= 1u;
            }
            G = __reduce_add_sync(kFull, G);
            bad = __reduce_or_sync(kFull, bad);
            const bool pass = bad == 0 && G < kBoundLimit;
            if (lane == l) {
                uint32_t* rec = g_out + (size_t)my_site * 32;
                rec[kWAlt] = pass ? 0u : my_act;
                // pass: single active allele REF, no EM ran: n_active 1, em_calls 0
                if (pass) rec[kWInfo] = (1u << 8) | (((my_info >> 16) & 0xffu) | BV_FLAG_LRT_BOUND) << 16;
                rec[kWState] = pass ? kStateDone : kStateEM;
                if (!pass) a.list_em[atomicAdd(a.counters + kCntEm, 1u)] = my_site;
            }
        }
    }
    grid_dep_launch();
}

// =====================================================================================================================
// K4: one warp per site of the EM list.
// =====================================================================================================================
constexpr int kQualWarps = 32;
constexpr int kP2Chunk = 512;                // cells per buffer and plane: kP2Chunk / 512 16-cell vectors per lane
constexpr int kP2Bufs = 2;                   // ring of row chunks per warp: kP2Bufs - 1 TMA fetches in flight ahead of the scan

struct __align__(128) P2Buf {                // one chunk of the base and qual planes
    uint8_t base[kP2Chunk];
    uint8_t qual[kP2Chunk];
};

struct __align__(128) QualWarp {
    P2Buf p2[kP2Bufs];
    uint32_t hist[kHistWords];   // (base, phred) histogram, all-zero between sites; the EM's per-bin state (one double
                                 // per compact bin) overlays it once the bins are compacted
    uint32_t bins[kSmemBins];    // compact non-empty bins: (base << 29) | (phred << 22) | count
    double emf[4];               // EM: allele frequencies in / out
    double res_f[4];             // LRT: frequencies of the accepted model
    double best_f[4];            // LRT: frequencies of the best candidate subset of the current round
    double res_chi;              // LRT: last chi_sqrt_value
    uint32_t flag_word;          // BV_FLAG_* raised inside out-of-line code
    uint32_t p2_phase;           // mbarrier phase bits of p2bar[]
    uint64_t p2bar[kP2Bufs];
    alignas(16) bv_site_out rec; // the site's record: loaded from global, completed, stored back
    uint32_t vcf_n;              // sites with ALT alleles waiting for their scalar finish (vcf_flush)
    uint32_t vcf_site[32];
};

struct __align__(128) QualCta {
    double lut[4 * kQStride];
    SiteKernelArgs a;            // kernel parameters for out-of-line device functions (a reference to the
                                 // __global__ parameter itself would force a local-memory copy)
};
constexpr size_t kQualSmemBytes = sizeof(QualCta) + (size_t)kQualWarps * sizeof(QualWarp);
static_assert(kQualSmemBytes <= 232448, "shared memory of the qual kernel exceeds 227 KB");

// K3's dynamic shared memory: QualCta, then one QualWarp per warp.
__device__ __forceinline__ QualCta& cta_shared() { return *reinterpret_cast<QualCta*>(bv_smem_raw); }
__device__ __forceinline__ QualWarp& warp_smem() {
    return reinterpret_cast<QualWarp*>(bv_smem_raw + sizeof(QualCta))[threadIdx.x >> 5];
}

__device__ __forceinline__ uint32_t pack_bin(uint32_t b, uint32_t q, uint32_t count) {
    return (b << 29) | (q << 22) | count;
}
__device__ __forceinline__ uint32_t bin_base(uint32_t p) { return p >> 29; }
__device__ __forceinline__ uint32_t bin_qual(uint32_t p) { return (p >> 22) & 0x7fu; }
__device__ __forceinline__ uint32_t bin_count(uint32_t p) { return p & 0x3fffffu; }

// ---- the row's base + qual chunks, fetched (L2 / HBM) into the warp's two buffers ---------------------------------------
// f(cellp, vb, lane_cells, cell0): cellp points at this lane's 16 base cells in shared memory (quals at cellp + kP2Chunk),
// vb holds them with padding cells masked to 'N', cell0 is the sample index of the first of them.
template <class F>
__device__ __forceinline__ void for_each_p2_chunk(uint32_t site, F&& f) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const int lane = threadIdx.x & 31;
    const uint32_t N = cs.a.n_samples;
    const uint32_t row_bytes = (N + 15u) & ~15u;
    const uint32_t nchunk = (row_bytes + kP2Chunk - 1) / kP2Chunk;
    const uint8_t* gb = cs.a.base + (size_t)site * cs.a.pitch;
    const uint8_t* gq = cs.a.qual + (size_t)site * cs.a.qual_pitch;
    const uint32_t s_buf0 = smem_u32(&W.p2[0]), s_bar0 = smem_u32(&W.p2bar[0]);
    uint32_t phase = W.p2_phase;
    auto fetch = [&](uint32_t c) {   // lane 0: chunk c into buffer c % kP2Bufs
        const uint32_t off = c * kP2Chunk;
        const uint32_t bytes = min((uint32_t)kP2Chunk, row_bytes - off);
        const uint32_t b = c % (uint32_t)kP2Bufs;
        const uint32_t bar = s_bar0 + 8u * b, dst = s_buf0 + (uint32_t)sizeof(P2Buf) * b;
        mbar_expect_tx(bar, 2 * bytes);
        bulk_g2s(dst, gb + off, bytes, bar);
        bulk_g2s(dst + kP2Chunk, gq + off, bytes, bar);
    };
    if (lane == 0) {
        for (uint32_t c = 0; c < (uint32_t)(kP2Bufs - 1) && c < nchunk; ++c) fetch(c);
    }
#pragma unroll 1
    for (uint32_t c = 0; c < nchunk; ++c) {
        const uint32_t buf = c % (uint32_t)kP2Bufs;
        // chunk c + kP2Bufs - 1 goes where chunk c - 1 was (all lanes are past it: __syncwarp below)
        if (c + (uint32_t)(kP2Bufs - 1) < nchunk && lane == 0) fetch(c + (uint32_t)(kP2Bufs - 1));
        mbar_wait(s_bar0 + 8u * buf, (phase >> buf) & 1u);
        phase ^= 1u << buf;
#pragma unroll 1
        for (int v = 0; v < kP2Chunk / 512; ++v) {
            const int lane_cells = (int)N - (int)(c * kP2Chunk) - v * 512 - lane * 16;
            if (v > 0 && (int)N - (int)(c * kP2Chunk) - v * 512 <= 0) break;   // (warp-uniform) the row ended in this chunk
            const uint8_t* cellp = W.p2[buf].base + v * 512 + lane * 16;
            uint4 vb = make_uint4(0x05050505u, 0x05050505u, 0x05050505u, 0x05050505u);
            if (lane_cells > 0) vb = *reinterpret_cast<const uint4*>(cellp);
            if (lane_cells < 16) mask_tail(vb, lane_cells);
            f(cellp, vb, lane_cells, c * kP2Chunk + v * 512 + lane * 16);
        }
        __syncwarp();
    }
    if (lane == 0) W.p2_phase = phase;
}

// phred range of the counted cells of W.hist as qmin | qmax << 8 | flags << 16 (qmin > qmax: no counted cell):
// lane l looks at slots l, l + 32, l + 64
__device__ __forceinline__ uint32_t hist_phred_range() {
    QualWarp& W = warp_smem();
    const int lane = threadIdx.x & 31;
    uint32_t nz[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int q = lane + 32 * r;
        nz[r] = W.hist[q] | W.hist[kQSlots + q] | W.hist[2 * kQSlots + q] | W.hist[3 * kQSlots + q] | W.hist[4 * kQSlots + q];
    }
    const uint32_t m0 = __ballot_sync(kFull, nz[0] != 0), m1 = __ballot_sync(kFull, nz[1] != 0), m2 = __ballot_sync(kFull, nz[2] != 0);
    uint32_t qmin = 0xffu, qmax = 0, flags = 0;
    if (m0 | m1 | m2) {
        qmin = m0 ? (uint32_t)__ffs(m0) - 1u : m1 ? 31u + (uint32_t)__ffs(m1) : 63u + (uint32_t)__ffs(m2);
        qmax = m2 ? 95u - (uint32_t)__clz(m2) : m1 ? 63u - (uint32_t)__clz(m1) : 31u - (uint32_t)__clz(m0);
    }
    if (qmax > BV_QUAL_MAX) flags |= BV_FLAG_BAD_QUAL;   // phred > 93: outside the reference's table (slots 94, 95)
    return qmin | (qmax << 8) | (flags << 16);
}

// (base, phred) histogram of the covered cells of one row into W.hist
// (BaseType::BaseType, src/basetype.cpp:45-71: one likelihood row per counted read, a function of base and phred only).
// Returns qmin | qmax << 8 | flags << 16 (qmin > qmax: no counted cell).
// grp != nullptr: only the samples of population group g are counted (__get_group_batchinfo,
// src/basetype_caller.cpp:781-797); grp[] is padded with BV_GROUP_NONE to a multiple of 16 entries.
//
// Two cell loops per 16-cell vector, chosen per vector by the fullest lane (warp-uniform):
//   sparse (< 1x pileups): the lane's counted cells one by one, found with bfind in its 16-bit mask; the warp runs as many
//     trips as its fullest lane has cells;
//   dense (deep pileups): all 16 cells straight from the registers that hold the vector, the mask bit as the predicate of
//     the shared-memory atomic: 5 instructions per cell instead of 10 per trip.
// The phred range is read off the histogram afterwards (96 slots, three per lane) instead of being tracked per cell.
constexpr int kHistDenseTrips = 7;   // the dense loop once the fullest lane of a vector has this many counted cells
// hist[idx] += 1 for the lanes with `on`, as ONE predicated instruction (no branch around it)
__device__ __forceinline__ void hist_add_if(uint32_t hist_s, uint32_t idx, uint32_t on) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.u32 p, %0, 0;\n\t"
        "@p red.shared.add.u32 [%1], 1;\n\t"
        "}" ::"r"(on), "r"(hist_s + 4u * idx) : "memory");
}
__device__ __forceinline__ void hist_word_dense(uint32_t hist_s, uint32_t wb, uint32_t wq, uint32_t t, int k) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t b = (wb >> (8 * j)) & 0xffu, q = (wq >> (8 * j)) & 0xffu;
        hist_add_if(hist_s, b * kQSlots + q, t & (1u << (8 * j + k)));
    }
}

__device__ __noinline__ uint32_t build_hist(uint32_t site, const uint8_t* grp, uint32_t g) {
    QualWarp& W = warp_smem();
    const uint32_t gw = g * 0x01010101u;
    for_each_p2_chunk(site, [&](const uint8_t* cellp, const uint4& vb, int lane_cells, uint32_t cell0) {
        // t: bit (8*j + k) set <=> byte j of word k holds a counted base code (< 5)
        uint32_t n0 = (((vb.x | 0x80808080u) - 0x05050505u) | vb.x) & 0x80808080u;
        uint32_t n1 = (((vb.y | 0x80808080u) - 0x05050505u) | vb.y) & 0x80808080u;
        uint32_t n2 = (((vb.z | 0x80808080u) - 0x05050505u) | vb.z) & 0x80808080u;
        uint32_t n3 = (((vb.w | 0x80808080u) - 0x05050505u) | vb.w) & 0x80808080u;
        if (grp != nullptr && lane_cells > 0) {   // cells of other groups are not counted (byte != g  =>  bit 7 set)
            const uint4 vg = __ldg(reinterpret_cast<const uint4*>(grp + cell0));
            uint32_t x;
            x = vg.x ^ gw; n0 |= (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
            x = vg.y ^ gw; n1 |= (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
            x = vg.z ^ gw; n2 |= (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
            x = vg.w ^ gw; n3 |= (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
        }
        uint32_t t = ((n0 >> 7) | (n1 >> 6) | (n2 >> 5) | (n3 >> 4)) ^ 0x0f0f0f0fu;
        // warp-uniform trip count, lanes that run out are predicated off: the warp never splits
        const int n = (int)__reduce_max_sync(kFull, (uint32_t)__popc(t));
        if (n >= kHistDenseTrips) {
            // phred > 95 shares the last slot (bytes >= 0x80 never occur next to a counted base in a valid tile; they clamp too)
            const uint4 vq = *reinterpret_cast<const uint4*>(cellp + kP2Chunk);
            const uint32_t hist_s = smem_u32(W.hist);
            hist_word_dense(hist_s, vb.x, __vminu4(vq.x, 0x5f5f5f5fu), t, 0);
            hist_word_dense(hist_s, vb.y, __vminu4(vq.y, 0x5f5f5f5fu), t, 1);
            hist_word_dense(hist_s, vb.z, __vminu4(vq.z, 0x5f5f5f5fu), t, 2);
            hist_word_dense(hist_s, vb.w, __vminu4(vq.w, 0x5f5f5f5fu), t, 3);
        } else {
#pragma unroll 1
            for (int i = 0; i < n; ++i) {
                const bool on = t != 0u;
                int top;
                asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(t));
                t &= ~(1u << (top & 31));
                const int cell = ((top & 3) << 2) | ((top >> 3) & 3);   // word k = top & 3, byte j = top >> 3
                if (on) {
                    const uint32_t b = cellp[cell];
                    const uint32_t q = min((uint32_t)cellp[cell + kP2Chunk], (uint32_t)(kQSlots - 1));   // phred > 95 shares the last slot
                    atomicAdd(&W.hist[b * kQSlots + q], 1u);
                }
            }
        }
    });
    __syncwarp();
    return hist_phred_range();
}

// ---- the same histogram for LONG rows (n_samples > kLongRowSamples): K4a only ------------------------------------------------
// A 100,000-sample row at 0.1x has 1.6 counted cells per 16-cell vector, but the warp runs as many trips of the cell loop as
// its FULLEST lane has cells (5 to 6): two thirds of the issue slots go to lanes that have run out.  Here a lane owns four
// vectors of a 2,048-cell chunk and walks one 64-bit mask of their 64 cells: the fullest of 32 lanes then has ~12 cells
// where the mean is 6.4, the fetch / wait / loop overhead of a chunk is paid once per four vectors, and the warp count
// per SM is halved to make room for the larger buffers (16 warps x 2 buffers x 4 KB).
constexpr int kLongWarps = 16;
constexpr int kLongVpl = 4;                   // 16-cell vectors per lane and chunk: 2 or 4
constexpr int kLongChunk = 512 * kLongVpl;    // cells per buffer and plane
static_assert(kLongVpl == 2 || kLongVpl == 4, "kLongVpl must be 2 or 4");
struct __align__(128) LongBuf {
    uint8_t base[kLongChunk];
    uint8_t qual[kLongChunk];
};
constexpr size_t kHistLongSmemBytes = sizeof(QualCta) + (size_t)kLongWarps * (sizeof(QualWarp) + 2 * sizeof(LongBuf));
static_assert(kHistLongSmemBytes <= 232448, "shared memory of the long-row histogram kernel exceeds 227 KB");
__device__ __forceinline__ LongBuf* long_bufs() {
    return reinterpret_cast<LongBuf*>(bv_smem_raw + sizeof(QualCta) + (size_t)kLongWarps * sizeof(QualWarp)) + 2 * (threadIdx.x >> 5);
}

// bit (4k + j) of the result: byte j of word k of the vector holds a counted base code (< 5)
__device__ __forceinline__ uint32_t counted_mask16(const uint4& vb) {
    const uint32_t w[4] = {vb.x, vb.y, vb.z, vb.w};
    uint32_t t = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t c = ~(((w[k] | 0x80808080u) - 0x05050505u) | w[k]) & 0x80808080u;   // bit 7 of every counted byte
        // the four bits 7, 15, 23, 31 land in bits 32..35 of the 64-bit product (all other partial products miss them)
        t |= (__umulhi(c, 0x02040810u) & 0xfu) << (4 * k);
    }
    return t;
}

__device__ __noinline__ uint32_t build_hist_long(uint32_t site) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    LongBuf* const LB = long_bufs();
    const int lane = threadIdx.x & 31;
    const uint32_t N = cs.a.n_samples;
    const uint32_t row_bytes = (N + 15u) & ~15u;
    const uint32_t nchunk = (row_bytes + kLongChunk - 1) / kLongChunk;
    const uint8_t* gb = cs.a.base + (size_t)site * cs.a.pitch;
    const uint8_t* gq = cs.a.qual + (size_t)site * cs.a.qual_pitch;
    const uint32_t s_buf0 = smem_u32(LB), s_bar0 = smem_u32(&W.p2bar[0]), hist_s = smem_u32(W.hist);
    uint32_t phase = W.p2_phase;
    auto fetch = [&](uint32_t c) {   // lane 0: chunk c into buffer c & 1
        const uint32_t off = c * kLongChunk;
        const uint32_t bytes = min((uint32_t)kLongChunk, row_bytes - off);
        const uint32_t b = c & 1u;
        const uint32_t bar = s_bar0 + 8u * b, dst = s_buf0 + (uint32_t)sizeof(LongBuf) * b;
        mbar_expect_tx(bar, 2 * bytes);
        bulk_g2s(dst, gb + off, bytes, bar);
        bulk_g2s(dst + kLongChunk, gq + off, bytes, bar);
    };
    if (lane == 0) fetch(0);
#pragma unroll 1
    for (uint32_t c = 0; c < nchunk; ++c) {
        const uint32_t buf = c & 1u;
        if (c + 1 < nchunk && lane == 0) fetch(c + 1);   // into the buffer chunk c - 1 used (all lanes are past it: __syncwarp below)
        mbar_wait(s_bar0 + 8u * buf, (phase >> buf) & 1u);
        phase ^= 1u << buf;
        const uint8_t* const cb = LB[buf].base + lane * 16;   // this lane's vector v is at cb + 512 v, its quals kLongChunk further
        // counted cells of this lane's vectors: vectors 0, 1 in lo (bit 16 v + cell), vectors 2, 3 in hi
        uint32_t lo = 0, hi = 0;
        uint4 vbs[kLongVpl];
#pragma unroll
        for (int v = 0; v < kLongVpl; ++v) {
            const int lane_cells = (int)N - (int)(c * kLongChunk) - v * 512 - lane * 16;
            uint4 vb = make_uint4(0x05050505u, 0x05050505u, 0x05050505u, 0x05050505u);
            if (lane_cells > 0) vb = *reinterpret_cast<const uint4*>(cb + 512 * v);
            if (lane_cells < 16) mask_tail(vb, lane_cells);
            vbs[v] = vb;
            const uint32_t tv = counted_mask16(vb) << (16 * (v & 1));
            if (v < 2) lo |= tv; else hi |= tv;
        }
        const int n = (int)__reduce_max_sync(kFull, (uint32_t)(__popc(lo) + __popc(hi)));
        if (n >= kLongVpl * kHistDenseTrips) {
#pragma unroll
            for (int v = 0; v < kLongVpl; ++v) {
                const uint4 vq = *reinterpret_cast<const uint4*>(cb + 512 * v + kLongChunk);
                const uint32_t wb[4] = {vbs[v].x, vbs[v].y, vbs[v].z, vbs[v].w};
                const uint32_t wq[4] = {__vminu4(vq.x, 0x5f5f5f5fu), __vminu4(vq.y, 0x5f5f5f5fu), __vminu4(vq.z, 0x5f5f5f5fu), __vminu4(vq.w, 0x5f5f5f5fu)};
                const uint32_t tv = ((v < 2 ? lo : hi) >> (16 * (v & 1))) & 0xffffu;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t b = (wb[k] >> (8 * j)) & 0xffu, q = (wq[k] >> (8 * j)) & 0xffu;
                        hist_add_if(hist_s, b * kQSlots + q, tv & (1u << (4 * k + j)));
                    }
                }
            }
        } else {
#pragma unroll 1
            for (int i = 0; i < n; ++i) {
                // this lane's next counted cell: from lo while it has any, then from hi (32-bit operations only)
                const bool in_lo = lo != 0u;
                const uint32_t w = in_lo ? lo : hi;
                int top;
                asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(w));
                const uint32_t rest = w & ~(1u << (top & 31));
                lo = in_lo ? rest : lo;
                hi = in_lo ? hi : rest;
                const int at = (in_lo ? 0 : 1024) + ((top & 16) << 5) + (top & 15);   // vector 2 * (hi) + (top >> 4), cell top & 15
                hist_add_if(hist_s, (uint32_t)cb[at & (kLongChunk - 1)] * kQSlots + min((uint32_t)cb[(at & (kLongChunk - 1)) + kLongChunk], (uint32_t)(kQSlots - 1)),
                            w != 0u);   // phred > 95 shares the last slot
            }
        }
        __syncwarp();
    }
    if (lane == 0) W.p2_phase = phase;
    __syncwarp();
    return hist_phred_range();
}

// ---- EM on compact bins (src/algorithm.h:210-255) ----------------------------------------------------------------
// bins: nb packed (base, phred, count) entries; lml: nb doubles of scratch (log marginal likelihood per bin).
// subset: bit j set => allele j in the candidate combination.  W.emf: initial frequencies in (NOT renormalised,
// src/basetype.cpp:93-103), estimated frequencies out.  Returns the sum of log marginal likelihoods under the
// second-to-last frequency vector, exactly what _f() sums (src/basetype.cpp:119-120).
// INT_SUM, the build for parameters away from the defaults (em_subset): BV_EM_ABS_INT_TRUNC with an eps outside (0, 1] compares
// EM()'s convergence sum itself, sum of count * (double)abs((int)diff) over the bins (see iabs_trunc), formed exactly in integers
// ("did some |diff| reach 1" answers "sum < eps" only for 0 < eps <= 1), and em_max_iter 0 runs no iteration.  Those EMs always
// take this build, so that the default build of it and em_bins_reg keep their registers.
template <bool INT_SUM>
__device__ __noinline__ double em_bins(const uint32_t* bins, double* lml, int nb, int subset, double total) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const double* s_lut = cs.lut;
    const int lane = threadIdx.x & 31;
    const int abs_mode = cs.a.abs_mode;
    double f0 = W.emf[0], f1 = W.emf[1], f2 = W.emf[2], f3 = W.emf[3];
    __syncwarp();
    int it = cs.a.em_max_iter;
    bool first = true;
    for (;;) {
        double s0 = 0, s1 = 0, s2 = 0, s3 = 0, delta = 0;
        long long isum = 0;
        bool big = false;
#pragma unroll 1
        for (int i = lane; i < nb; i += 32) {
            const uint32_t p = bins[i];
            const uint32_t b = bin_base(p), q = bin_qual(p);
            const double cd = (double)bin_count(p);
            const double ome = s_lut[kLutOneMinusEps * kQStride + q], e3 = s_lut[kLutEpsThird * kQStride + q];
            // e_step (algorithm.h:160-172): lik*freq summed in A,C,G,T order; alleles outside the subset have
            // freq 0 and add an exact +0.0, so they are skipped
            double l0 = 0, l1 = 0, l2 = 0, l3 = 0, m = 0;
            if (subset & 1) { l0 = (b == 0 ? ome : e3) * f0; m += l0; }
            if (subset & 2) { l1 = (b == 1 ? ome : e3) * f1; m += l1; }
            if (subset & 4) { l2 = (b == 2 ? ome : e3) * f2; m += l2; }
            if (subset & 8) { l3 = (b == 3 ? ome : e3) * f3; m += l3; }
            const double llh = log(m);
            if (!first) {
                const double diff = llh - lml[i];
                if (abs_mode == BV_EM_ABS_INT_TRUNC) {
                    // (double)abs((int)diff): non-zero iff |diff| >= 1; NaN/inf convert to INT_MIN whose
                    // "abs" stays negative and ends the loop (results are NaN by then)
                    if (INT_SUM) isum += (long long)bin_count(p) * iabs_trunc(diff);
                    else if (fabs(diff) >= 1.0 && fabs(diff) < 2147483648.0) big = true;
                } else {
                    delta += cd * fabs(diff);
                }
            }
            lml[i] = llh;
            // m_step (algorithm.h:184-198): column sums of the posteriors; c equal reads add c * post
            if (subset & 1) s0 += cd * (l0 / m);
            if (subset & 2) s1 += cd * (l1 / m);
            if (subset & 4) s2 += cd * (l2 / m);
            if (subset & 8) s3 += cd * (l3 / m);
        }
        if (subset & 1) f0 = warp_sum(s0) / total;
        if (subset & 2) f1 = warp_sum(s1) / total;
        if (subset & 4) f2 = warp_sum(s2) / total;
        if (subset & 8) f3 = warp_sum(s3) / total;
        if (first) {
            first = false;
            if (!INT_SUM || it != 0) continue;
            // em_max_iter 0: while (it--) { ... } (src/algorithm.h:234-251) runs no iteration after the first E-step + M-step
            if (lane == 0) W.flag_word |= BV_FLAG_EM_MAXITER;
            break;
        }
        bool more;
        if (abs_mode != BV_EM_ABS_INT_TRUNC) more = !(warp_sum(delta) < cs.a.em_eps);
        else if (INT_SUM) more = !((double)warp_sum_ll(isum) < cs.a.em_eps);
        else more = __any_sync(kFull, big);
        --it;
        if (it == 0 && lane == 0) W.flag_word |= BV_FLAG_EM_MAXITER;
        if (!more || it == 0) break;
    }
    double ll = 0;
#pragma unroll 1
    for (int i = lane; i < nb; i += 32) ll += (double)bin_count(bins[i]) * lml[i];
    if (lane == 0) { W.emf[0] = f0; W.emf[1] = f1; W.emf[2] = f2; W.emf[3] = f3; }
    __syncwarp();
    return warp_sum(ll);
}

// ---- the same EM with the bins in registers ------------------------------------------------------------------------
// Up to 32 * NS bins: lane l owns bins l, l + 32, ... (the order em_bins visits them in, so every sum is associated the
// same way).  Each lane keeps its bins' likelihoods, counts and previous marginals in registers over all iterations and
// works on its NS bins in one straight-line block, so that NS independent FP64 chains are in flight.  Two savings in
// operation count, both inside the stated tolerance of the floating-point outputs (1e-9 here, 1e-6 in north_star):
//   * the four posteriors of a read are l_j * (1/m) instead of l_j / m: one division per bin instead of one per allele;
//   * as built (int abs(int), src/algorithm.h:245) the convergence sum is non-zero only when some log-marginal moved by
//     at least 1, i.e. when a marginal changed by a factor e: decided exactly from the ratio of the marginals -- inside
//     (1/2.5, 2.5) no logarithm is needed, otherwise the logarithms themselves decide -- so that `log` runs once per
//     bin and EM call (for the reported log-likelihoods) instead of once per bin and iteration.
// Logarithms through nlog, out of line: the inlined libdevice log is ~90 instructions per call site and this kernel is
// instruction-fetch sensitive.
template <int NS>
__device__ __noinline__ double em_bins_reg(const uint32_t* bins, int nb, int subset, double total) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const double* s_lut = cs.lut;
    const int lane = threadIdx.x & 31;
    const bool int_mode = cs.a.abs_mode == BV_EM_ABS_INT_TRUNC;
    double f0 = W.emf[0], f1 = W.emf[1], f2 = W.emf[2], f3 = W.emf[3];
    __syncwarp();
    double ome[NS], e3[NS], cd[NS], prev[NS];   // prev: marginal (int mode) or log marginal (double mode) of the last E-step
    uint32_t bb[NS];
    bool on[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const int i = lane + 32 * k;
        on[k] = i < nb;
        const uint32_t p = on[k] ? bins[i] : pack_bin(4u, 0u, 0u);
        const uint32_t q = bin_qual(p);
        bb[k] = bin_base(p);
        cd[k] = (double)bin_count(p);
        ome[k] = s_lut[kLutOneMinusEps * kQStride + q];
        e3[k] = s_lut[kLutEpsThird * kQStride + q];
        prev[k] = 0.0;
    }
    int it = cs.a.em_max_iter;
    bool first = true;
    for (;;) {
        double s0 = 0, s1 = 0, s2 = 0, s3 = 0, delta = 0;
        bool big = false, unsure = false;
        double mk[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            // e_step (algorithm.h:160-172): lik*freq summed in A,C,G,T order; alleles outside the subset add an exact +0.0
            double l0 = 0, l1 = 0, l2 = 0, l3 = 0, m = 0;
            if (subset & 1) { l0 = (bb[k] == 0 ? ome[k] : e3[k]) * f0; m += l0; }
            if (subset & 2) { l1 = (bb[k] == 1 ? ome[k] : e3[k]) * f1; m += l1; }
            if (subset & 4) { l2 = (bb[k] == 2 ? ome[k] : e3[k]) * f2; m += l2; }
            if (subset & 8) { l3 = (bb[k] == 3 ? ome[k] : e3[k]) * f3; m += l3; }
            mk[k] = m;
            const double inv = 1.0 / m;
            // m_step (algorithm.h:184-198): column sums of the posteriors; c equal reads add c * post
            if (on[k]) {
                if (subset & 1) s0 += cd[k] * (l0 * inv);
                if (subset & 2) s1 += cd[k] * (l1 * inv);
                if (subset & 4) s2 += cd[k] * (l2 * inv);
                if (subset & 8) s3 += cd[k] * (l3 * inv);
            }
        }
        if (int_mode) {
            if (!first) {
#pragma unroll
                for (int k = 0; k < NS; ++k)
                    if (on[k] && !(mk[k] < 2.5 * prev[k] && prev[k] < 2.5 * mk[k])) unsure = true;   // also NaN / 0 / inf
                if (__any_sync(kFull, unsure)) {
#pragma unroll
                    for (int k = 0; k < NS; ++k) {
                        // (double)abs((int)diff): non-zero iff |diff| >= 1; NaN/inf convert to INT_MIN whose "abs" stays
                        // negative and ends the loop (results are NaN by then)
                        const double diff = nlog(mk[k]) - nlog(prev[k]);
                        if (on[k] && fabs(diff) >= 1.0 && fabs(diff) < 2147483648.0) big = true;
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < NS; ++k) prev[k] = mk[k];
        } else {
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                const double llh = nlog(mk[k]);
                if (!first && on[k]) delta += cd[k] * fabs(llh - prev[k]);
                prev[k] = llh;
            }
        }
        if (subset & 1) f0 = warp_sum(s0) / total;
        if (subset & 2) f1 = warp_sum(s1) / total;
        if (subset & 4) f2 = warp_sum(s2) / total;
        if (subset & 8) f3 = warp_sum(s3) / total;
        if (first) { first = false; continue; }
        bool more;
        if (int_mode) more = __any_sync(kFull, big);
        else more = !(warp_sum(delta) < cs.a.em_eps);
        --it;
        if (it == 0 && lane == 0) W.flag_word |= BV_FLAG_EM_MAXITER;
        if (!more || it == 0) break;
    }
    double ll = 0;
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const double lml = int_mode ? nlog(prev[k]) : prev[k];
        if (on[k]) ll += cd[k] * lml;
    }
    if (lane == 0) { W.emf[0] = f0; W.emf[1] = f1; W.emf[2] = f2; W.emf[3] = f3; }
    __syncwarp();
    return warp_sum(ll);
}

// EM of one candidate subset: bins in registers when they fit (the usual case), else the loop over memory
__device__ __forceinline__ double em_subset(const uint32_t* bins, double* lml, int nb, int subset, double total) {
    const SiteKernelArgs& a = cta_shared().a;
    if ((a.abs_mode == BV_EM_ABS_INT_TRUNC && !(a.em_eps > 0.0 && a.em_eps <= 1.0)) || a.em_max_iter == 0)
        return em_bins<true>(bins, lml, nb, subset, total);
    if (nb <= 32) return em_bins_reg<1>(bins, nb, subset, total);
    if (nb <= 96) return em_bins_reg<3>(bins, nb, subset, total);
    return em_bins<false>(bins, lml, nb, subset, total);
}

// Log-likelihood of the single-allele model {b} (an EM whose answer is closed form):
// after the first m_step f_b == 1.0 exactly (every posterior is x/x), so every later marginal is L_b itself and
// the reported log marginal is log(1-eps) or log(eps/3) -- both tabulated on the host with glibc.  A bin of base b
// with phred 0 has L_b == 0: the reference then divides 0/0 and everything becomes NaN (returned as NaN).
__device__ __noinline__ double single_allele_ll(const uint32_t* bins, int nb, int b_allele) {
    const double* s_lut = cta_shared().lut;
    const int lane = threadIdx.x & 31;
    double ll = 0;
    bool bad = false;
#pragma unroll 1
    for (int i = lane; i < nb; i += 32) {
        const uint32_t p = bins[i];
        const uint32_t b = bin_base(p), q = bin_qual(p);
        const bool match = ((int)b == b_allele);
        if (match && q == 0) bad = true;
        ll += (double)bin_count(p) * s_lut[(match ? kLutLogMatch : kLutLogMis) * kQStride + q];
    }
    ll = warp_sum(ll);
    if (__any_sync(kFull, bad)) ll = __longlong_as_double(0x7ff8000000000000ll);
    return ll;
}

// The same for all four bases in one pass over the bins: out[b] is, bit for bit, single_allele_ll(bins, nb, b) (every lane sums
// the same bins in the same order, the lanes' sums meet in the same butterfly).  K4a leaves them with the site's header, so the
// thread that later decides the site needs no pass over the bins.
__device__ __noinline__ void single_allele_ll4(const uint32_t* bins, int nb, double (&out)[4]) {
    const double* s_lut = cta_shared().lut;
    const int lane = threadIdx.x & 31;
    double ll[4] = {0, 0, 0, 0};
    uint32_t bad = 0;
#pragma unroll 1
    for (int i = lane; i < nb; i += 32) {
        const uint32_t p = bins[i];
        const uint32_t b = bin_base(p), q = bin_qual(p);
        const double c = (double)bin_count(p);
        const double lm = s_lut[kLutLogMatch * kQStride + q], lx = s_lut[kLutLogMis * kQStride + q];
        if (q == 0 && b < 4u) bad |= 1u << b;
#pragma unroll
        for (int k = 0; k < 4; ++k) ll[k] += c * ((int)b == k ? lm : lx);
    }
    bad = __reduce_or_sync(kFull, bad);
    // warp_sum's butterfly, the four sums side by side (four independent chains instead of four calls one after the other)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 4; ++k) ll[k] += __shfl_xor_sync(kFull, ll[k], o);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) out[k] = (bad >> k & 1u) ? __longlong_as_double(0x7ff8000000000000ll) : ll[k];
}

// The k-th (k >= 0) active base of an ORDERED base list: `order` packs the list two bits per position (position 0 in
// bits 0-1), `mask` says which alleles are active.  BaseType::lrt() passes A,C,G,T (kOrderACGT); the population-group
// calls pass [REF, ALT...] (src/basetype_caller.cpp:750-753), and the order decides which subset wins a tie and which
// base is dropped first (src/external/combinations.h:19-84).
constexpr uint32_t kOrderACGT = 0xE4u;
__device__ __forceinline__ int nth_active(uint32_t order, uint32_t mask, int k) {
    int pos = -1;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        const int b = (int)((order >> (2 * p)) & 3u);
        if (mask & (1u << b)) {
            if (k == 0 && pos < 0) pos = b;
            --k;
        }
    }
    return pos;
}

// ---- sites with >= 2 active alleles: compact the bins, EM on the full set, backward elimination -----------------------
// (src/basetype.cpp:144-168).  In: the row's histogram in W.hist, phred range, depths in W.rec.depth[], active set.
// Out: W.res_f / W.res_chi and the return value act | n_act << 4 | em_calls << 8.  The warp-uniform model state lives
// in shared memory (W.emf / W.best_f / W.res_f), not in registers that would have to survive the calls into em_bins.

// The non-empty (base, phred) bins of W.hist, in (base, phred) order, into W.bins (the first kSmemBins of them) and into
// this warp's global spill row (all of them); the histogram goes back to zero.  Returns the number of bins.
__device__ __noinline__ int compact_bins(uint32_t qmin, uint32_t qmax) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const int lane = threadIdx.x & 31;
    const uint32_t warp_global = blockIdx.x * kQualWarps + (threadIdx.x >> 5);
    int nb = 0;
    uint32_t* gbins = cs.a.bin_spill + (size_t)warp_global * kMaxBins;
#pragma unroll 1
    for (int b = 0; b < 5; ++b) {
        if (b < 4 ? W.rec.depth[b] == 0 : W.rec.depth_other == 0) continue;
#pragma unroll 1
        for (uint32_t q0 = qmin; q0 <= qmax; q0 += 32) {
            const uint32_t q = q0 + lane;
            uint32_t v = 0;
            if (q <= qmax) {
                v = W.hist[b * kQSlots + q];
                W.hist[b * kQSlots + q] = 0;
            }
            const uint32_t bal = __ballot_sync(kFull, v != 0);
            if (v) {
                const int pos = nb + __popc(bal & ((1u << lane) - 1u));
                const uint32_t p = pack_bin(b, q, v);
                if (pos < kSmemBins) W.bins[pos] = p;
                gbins[pos] = p;
            }
            nb += __popc(bal);
        }
    }
    __syncwarp();
    return nb;
}

__device__ __noinline__ uint32_t lrt_on_bins(int nb, uint32_t act, uint32_t order) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const int lane = threadIdx.x & 31;
    const uint32_t warp_global = blockIdx.x * kQualWarps + (threadIdx.x >> 5);
    uint32_t* gbins = cs.a.bin_spill + (size_t)warp_global * kMaxBins;
    // bins live in shared memory unless there are more than kSmemBins of them (then the global copy is used);
    // the EM's per-bin state overlays the (now all-zero) histogram
    const bool in_smem = nb <= kSmemBins;
    const uint32_t* bins = in_smem ? W.bins : gbins;
    double* lml = in_smem ? reinterpret_cast<double*>(W.hist) : cs.a.lml_spill + (size_t)warp_global * kMaxBins;

    const double dtot = (double)(W.rec.depth[0] + W.rec.depth[1] + W.rec.depth[2] + W.rec.depth[3] + W.rec.depth_other);
    int n_act = __popc(act);
    uint32_t flags = 0;
    double chi = 0.0;
    // initial frequencies of a subset: depth/total for its members, 0 elsewhere (src/basetype.cpp:93-103)
    if (lane < 4) W.emf[lane] = (act >> lane & 1u) ? (double)W.rec.depth[lane] / dtot : 0.0;
    __syncwarp();
    double lr_alt = em_subset(bins, lml, nb, (int)act, dtot);
    if (lane < 4) W.res_f[lane] = W.emf[lane];
    uint32_t em_calls = 1;
#pragma unroll 1
    for (int n = n_act - 1; n > 0; --n) {
        // the n-subsets of the n+1 active bases in the lexicographic order of
        // src/external/combinations.h:19-84: the i-th subset drops the (n-i)-th active base
        double best_chi = 0, best_lr = 0;
        uint32_t best_set = 0;
#pragma unroll 1
        for (int i = 0; i <= n; ++i) {
            const uint32_t sub = act & ~(1u << nth_active(order, act, n - i));
            __syncwarp();
            if (lane < 4) W.emf[lane] = (sub >> lane & 1u) ? (double)W.rec.depth[lane] / dtot : 0.0;
            __syncwarp();
            if (W.emf[0] + W.emf[1] + W.emf[2] + W.emf[3] == 0) flags |= BV_FLAG_ZERO_SUBSET;   // the reference throws (basetype.cpp:113)
            double lr;
            if (n == 1) {
                const int single = __ffs(sub) - 1;
                flags |= single_em_flag(W.rec.depth[single], (uint32_t)dtot, cs.a);
                lr = single_allele_ll(bins, nb, single);
                if (cs.a.em_max_iter == 0) lr += first_estep_ll_shift(W.rec.depth[single], dtot);
                const double v = (lr != lr) ? lr : 1.0;
                __syncwarp();   // every lane has read W.emf above
                if (lane < 4) W.emf[lane] = lane == single ? v : 0.0;
                __syncwarp();
            } else {
                lr = em_subset(bins, lml, nb, (int)sub, dtot);
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
                if (lane < 4) W.best_f[lane] = W.emf[lane];
            }
        }
        lr_alt = best_lr;
        chi = best_chi;
        const double lrt_threshold = cs.a.lrt_threshold;
        if (fabs(chi - lrt_threshold) < 1e-9 * lrt_threshold) flags |= BV_FLAG_NEAR_LRT;
        if (chi < lrt_threshold) {
            act = best_set; n_act = n;
            __syncwarp();
            if (lane < 4) W.res_f[lane] = W.best_f[lane];
        } else {
            break;
        }
    }
    // the EM state overlaid the histogram: back to all-zero for the next site
    __syncwarp();
    if (in_smem) {
#pragma unroll 1
        for (int i = lane; i < 2 * nb; i += 32) W.hist[i] = 0;
    }
    if (lane == 0) {
        W.res_chi = chi;
        W.flag_word |= flags;
    }
    __syncwarp();
    return act | ((uint32_t)n_act << 4) | (em_calls << 8);
}

__device__ __forceinline__ uint32_t lrt_multi(uint32_t qmin, uint32_t qmax, uint32_t act, uint32_t order) {
    const int nb = compact_bins(qmin, qmax);
    return lrt_on_bins(nb, act, order);
}

// ---- scalar finish of the sites with ALT alleles, one THREAD per queued site ------------------------------------------------
// QUAL = -10 log10 of the chi-square survival function of the last LRT statistic (src/basetype.cpp:188-194) unless the
// mono-allelic rule already set it, and the strand bias of the VCF row, ref vs the called ALT alleles
// (src/basetype.cpp:244-295, basetype_caller.cpp:1164).  Both are functions of a few numbers of the record; done inside
// qual_site the whole warp would compute them 32 times over (34 % of K4's instructions on C5 before this queue).
__device__ __noinline__ void vcf_flush() {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n = W.vcf_n;
    __syncwarp();
    bool job = false, wide = false;
    uint32_t entry = 0;
    if (lane < n) {
        const uint32_t site = W.vcf_site[lane];
        bv_site_out* rec = cs.a.out + site;
        const int ref_code = ref_code_of(cs.a.ref_base[site]);
        if (!(rec->flags & BV_FLAG_MONO_QUAL)) rec->qual = qual_from_chi(rec->chi2);
        uint32_t alt_set = 0;
        for (int k = 0; k < (int)rec->n_alt; ++k) alt_set |= 1u << (rec->alt[k] & 3u);
        int rf, rr, vf, vr, af_, ar;
        strand_tables(rec, ref_code, alt_set, rf, rr, vf, vr, af_, ar);
        double fs_vcf = 0.0;
        if ((vf | vr) != 0 && (rf | rr) != 0) {
            double p;
            if (fisher_margin1(rf, rr, vf, vr, p)) fs_vcf = fs_from_p(p);
            else { job = true; wide = fisher_support_wide(rf, rr, vf, vr); }   // bv_fisher_kernel completes the record
        }
        rec->fs_vcf = fs_vcf;
        entry = site | kFisherVcfRow;
    }
    fisher_push(cs.a, job, wide, entry);
    __syncwarp();
    if (lane == 0) W.vcf_n = 0;
    __syncwarp();
}

}  // namespace bv
