// bv_call_kernels.cuh -- the kernels of the CALLED sites (n_alt > 0), the rows of the VCF file.
//
//   K5  bv_ranksum_kernel  one warp per called site: the three rank-sum INFO fields of `_out_vcf_line`
//        (src/basetype_caller.cpp:1151-1157): ref_vs_alt_ranksumtest (src/basetype.cpp:201-242) over the mapping
//        qualities, the read position ranks and the base qualities of REF reads vs reads of the called ALT alleles,
//        each a Wilcoxon rank-sum test with a normal approximation (src/algorithm.h:48-50,76-136, kf_erfc
//        htslib/kfunc.c:58-84), phred scaled and truncated to int.
//   K6  bv_group_kernel    one warp per (called site, population group): `__gb` (src/basetype_caller.cpp:767-797) =
//        BaseType over the group's samples + lrt([upper REF, ALT...]); its ALT list and AFs (the "<group>_AF=" entries
//        of the INFO field, src/basetype_caller.cpp:1184-1194).  Reuses K4's histogram / EM / LRT code.
//
// Both take the called sites from the list K4 appends to.  A few per mille of the sites are called at 0.1x, so the
// four planes of a row are fetched (TMA bulk copies, from HBM or in place from pinned host memory) only here.
#pragma once
#include "bv_finish_kernels.cuh"

namespace bv {

// =====================================================================================================================
// K5: rank sums.
//
// wilcoxon_ranksum_test sorts the pooled values in DESCENDING order, gives ties their average rank and sums the ranks
// of sample 1 (the REF reads).  Ranks are half-integers and every partial sum is exact in FP64, so the sum does not
// depend on the order of the operations and is a function of the per-value class counts r(v), a(v):
//     2 * smp1_ranksum = sum_v r(v) * (2 * G(v) + t(v) + 1),   t = r + a,   G(v) = sum_{u > v} t(u)
// which is what the warp computes, in integers, from per-class value histograms in shared memory.  Mapping and base
// qualities are bytes; read position ranks up to kRprBins - 1 (short reads) use a histogram too, larger ones (long
// reads) fall back to pairwise counting, which is exact for any value.
// =====================================================================================================================
constexpr int kCallWarps = 8;
constexpr int kCChunk = 512;       // cells per buffer and plane, one 16-cell vector per lane
constexpr int kRprBins = 1024;

struct __align__(128) CallBuf {
    uint8_t base[kCChunk];
    uint8_t qual[kCChunk];
    uint8_t mapq[kCChunk];
    uint16_t rpr[kCChunk];
};
struct __align__(128) CallWarp {
    CallBuf buf[2];
    uint32_t h_mq[2][256];         // [class: 0 REF, 1 ALT][value], all-zero between sites
    uint32_t h_bq[2][256];
    uint32_t h_rp[2][kRprBins];
    uint64_t bar[2];
};
constexpr size_t kCallSmemBytes = (size_t)kCallWarps * sizeof(CallWarp);
static_assert(kCallSmemBytes <= 232448, "shared memory of the rank-sum kernel exceeds 227 KB");

// kf_erfc, htslib/kfunc.c:58-84 (AS66), operation by operation
__device__ __noinline__ double erfc_as66(double x) {
    const double p0 = 220.2068679123761, p1 = 221.2135961699311, p2 = 112.0792914978709, p3 = 33.912866078383,
                 p4 = 6.37396220353165, p5 = .7003830644436881, p6 = .03526249659989109;
    const double q0 = 440.4137358247522, q1 = 793.8265125199484, q2 = 637.3336333788311, q3 = 296.5642487796737,
                 q4 = 86.78073220294608, q5 = 16.06417757920695, q6 = 1.755667163182642, q7 = .08838834764831844;
    const double sqrt2 = 1.41421356237309504880;   // M_SQRT2
    double expntl, z, p;
    z = fabs(x) * sqrt2;
    if (z > 37.) return x > 0. ? 0. : 2.;
    expntl = nexp(z * z * -.5);
    if (z < 10. / sqrt2)
        p = expntl * ((((((p6 * z + p5) * z + p4) * z + p3) * z + p2) * z + p1) * z + p0) /
            (((((((q7 * z + q6) * z + q5) * z + q4) * z + q3) * z + q2) * z + q1) * z + q0);
    else
        p = expntl / 2.506628274631001 / (z + 1. / (z + 2. / (z + 3. / (z + 4. / (z + .65)))));
    return x > 0. ? 2. * p : 2. * (1. - p);
}

// From 2 * smp1_ranksum to the value of ref_vs_alt_ranksumtest: src/algorithm.h:130-135, src/basetype.cpp:224-236
// (n1, n2 > 0).  The sign of a zero result is left as the arithmetic gives it (-0.0 when every value ties).
__device__ __noinline__ double ranksum_phred_double(unsigned long long twice_ranksum, unsigned long long n1,
                                                    unsigned long long n2) {
    const double smp1_ranksum = (double)twice_ranksum / 2.0;
    const double e = (double)(n1 * (n1 + n2 + 1)) / 2.0;
    const double z = (smp1_ranksum - e) / sqrt((double)(n1 * n2 * (n1 + n2 + 1)) / 12.0);
    const double nd = erfc_as66(fabs(z) / sqrt(2.0)) / 2.0;   // norm_dist(std::abs(z))
    const double p = 2 * nd;
    double v = -10 * nlog10(p);
    if (isinf(v)) v = 10000;
    return v;
}

// the INFO value: (int) at src/basetype_caller.cpp:1151-1157
__device__ __noinline__ int ranksum_phred(unsigned long long twice_ranksum, unsigned long long n1, unsigned long long n2) {
    return (int)ranksum_phred_double(twice_ranksum, n1, n2);
}

// 2 * (rank sum of class 0) from the two class histograms over bins [vmin, vmax] (a larger bin is a larger value); the bins
// are zeroed on the way.  above_io (optional): reads with a value above bin vmax on entry, all reads counted so far on exit.
__device__ __forceinline__ unsigned long long hist_twice_ranksum(uint32_t* h0, uint32_t* h1, int vmin, int vmax,
                                                                 unsigned long long* above_io = nullptr) {
    const int lane = threadIdx.x & 31;
    unsigned long long acc = 0, above = above_io ? *above_io : 0ull;   // above: reads with a value greater than this step's 32 bins
#pragma unroll 1
    for (int top = vmax; top >= vmin; top -= 32) {
        const int v = top - lane;
        uint32_t r = 0, a = 0;
        if (v >= vmin) {
            r = h0[v]; a = h1[v];
            h0[v] = 0; h1[v] = 0;
        }
        const uint32_t t = r + a;
        uint32_t incl = t;   // inclusive scan over the lanes (lane 0 holds the largest value)
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += y;
        }
        const unsigned long long G = above + (incl - t);
        acc += (unsigned long long)r * (2ull * G + t + 1ull);
        above += __shfl_sync(kFull, incl, 31);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
    if (above_io) *above_io = above;
    return acc;
}

// class of a base code: 0 REF, 1 called ALT, 2 neither (src/basetype.cpp:211-220)
__device__ __forceinline__ uint32_t call_class(uint32_t b, int ref_code, uint32_t alt_mask) {
    if (b > 3u) return 2u;
    if ((int)b == ref_code) return 0u;
    return (alt_mask >> b) & 1u ? 1u : 2u;
}

struct CallKernelRow {
    const uint8_t *gb, *gq, *gm;
    const uint16_t* gr;
    uint32_t row_bytes, nchunk;
};

// issue the TMA copies of chunk c of a row into buffer `buf` (lane 0 only)
__device__ __forceinline__ void call_issue(CallWarp& W, const CallKernelRow& R, uint32_t c, uint32_t buf, bool with_qm) {
    const uint32_t off = c * kCChunk;
    const uint32_t bytes = min((uint32_t)kCChunk, R.row_bytes - off);
    const uint32_t bar = smem_u32(&W.bar[buf]), dst = smem_u32(&W.buf[buf]);
    mbar_expect_tx(bar, (with_qm ? 5u : 3u) * bytes);
    bulk_g2s(dst, R.gb + off, bytes, bar);
    if (with_qm) {
        bulk_g2s(dst + kCChunk, R.gq + off, bytes, bar);
        bulk_g2s(dst + 2 * kCChunk, R.gm + off, bytes, bar);
    }
    bulk_g2s(dst + 3 * kCChunk, R.gr + off, 2u * bytes, bar);
}

// Pairwise fallback for read position ranks >= kRprBins: 2 * smp1_ranksum = sum over REF reads i of
// (2 * #{j: v_j > v_i} + #{j: v_j == v_i} + 1), j over REF and ALT reads (i included).  Chunk A holds the REF reads a
// lane owns, chunk B sweeps the row.  Rare (long reads only); exact for any value.
__device__ __noinline__ unsigned long long rpr_pairwise(CallWarp& W, const CallKernelRow& R, uint32_t N, int ref_code,
                                                       uint32_t alt_mask, uint32_t& phase) {
    const int lane = threadIdx.x & 31;
    unsigned long long acc = 0;
#pragma unroll 1
    for (uint32_t ca = 0; ca < R.nchunk; ++ca) {
        if (lane == 0) call_issue(W, R, ca, 0, false);
        mbar_wait(smem_u32(&W.bar[0]), phase & 1u);
        phase ^= 1u;
        // this lane's REF reads of chunk A
        uint32_t mine = 0;
        uint16_t va[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const uint32_t i = ca * kCChunk + lane * 16 + k;
            va[k] = W.buf[0].rpr[lane * 16 + k];
            if (i < N && call_class(W.buf[0].base[lane * 16 + k], ref_code, alt_mask) == 0u) mine |= 1u << k;
        }
        const bool any = __any_sync(kFull, mine != 0u);
        if (any) {
#pragma unroll 1
            for (uint32_t cb = 0; cb < R.nchunk; ++cb) {
                if (lane == 0) call_issue(W, R, cb, 1, false);
                mbar_wait(smem_u32(&W.bar[1]), (phase >> 1) & 1u);
                phase ^= 2u;
                const uint32_t cells = min((uint32_t)kCChunk, N - cb * kCChunk);
#pragma unroll 1
                for (uint32_t j = 0; j < cells; ++j) {
                    if (call_class(W.buf[1].base[j], ref_code, alt_mask) == 2u) continue;   // warp-uniform
                    const uint32_t vj = W.buf[1].rpr[j];
#pragma unroll
                    for (int k = 0; k < 16; ++k)
                        if (mine >> k & 1u) acc += vj > va[k] ? 2ull : (vj == va[k] ? 1ull : 0ull);
                }
                __syncwarp();
            }
        }
        acc += (unsigned long long)__popc(mine);
        __syncwarp();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
    return acc;
}

__global__ void __launch_bounds__(kCallWarps * 32, 1) bv_ranksum_kernel(const __grid_constant__ SiteKernelArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    CallWarp& W = reinterpret_cast<CallWarp*>(bv_smem_raw)[warp];
    for (int i = lane; i < 2 * 256; i += 32) { (&W.h_mq[0][0])[i] = 0; (&W.h_bq[0][0])[i] = 0; }
    for (int i = lane; i < 2 * kRprBins; i += 32) (&W.h_rp[0][0])[i] = 0;
    if (lane == 0) {
        mbar_init(&W.bar[0], 1);
        mbar_init(&W.bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint32_t N = a.n_samples;
    const uint32_t n_called = a.counters[kCntCalled];
    const uint32_t total_warps = gridDim.x * kCallWarps;
    uint32_t phase = 0;   // bit b: parity of bar[b]
    CallKernelRow R;
    R.row_bytes = (N + 15u) & ~15u;
    R.nchunk = (R.row_bytes + kCChunk - 1) / kCChunk;

#pragma unroll 1
    for (uint32_t k = blockIdx.x * kCallWarps + warp; k < n_called; k += total_warps) {
        const uint32_t site = a.list_called[k];
        const uint32_t* rec = reinterpret_cast<const uint32_t*>(a.out + site);
        // n_alt, alt[0..2] in word kWAlt, alt[3] in the low byte of word kWInfo
        const uint32_t w_alt = rec[kWAlt], w_info = rec[kWInfo];
        const uint32_t n_alt = w_alt & 0xffu;
        uint32_t alt_mask = 0;
        if (n_alt > 0) alt_mask |= 1u << ((w_alt >> 8) & 3u);
        if (n_alt > 1) alt_mask |= 1u << ((w_alt >> 16) & 3u);
        if (n_alt > 2) alt_mask |= 1u << ((w_alt >> 24) & 3u);
        if (n_alt > 3) alt_mask |= 1u << (w_info & 3u);
        const int ref_code = ref_code_of(a.ref_base[site]);
        R.gb = a.base + (size_t)site * a.pitch;
        R.gq = a.qual + (size_t)site * a.qual_pitch;
        R.gm = a.mapq + (size_t)site * a.aux_pitch;
        R.gr = a.rpr + (size_t)site * a.rpr_pitch;

        uint32_t cnt0 = 0, cnt1 = 0;
        uint32_t mq_lo = 255, mq_hi = 0, bq_lo = 255, bq_hi = 0, rp_lo = 0xffffu, rp_hi = 0;
        if (lane == 0) call_issue(W, R, 0, 0, true);
#pragma unroll 1
        for (uint32_t c = 0; c < R.nchunk; ++c) {
            const uint32_t buf = c & 1u;
            if (c + 1 < R.nchunk && lane == 0) call_issue(W, R, c + 1, buf ^ 1u, true);
            mbar_wait(smem_u32(&W.bar[buf]), (phase >> buf) & 1u);
            phase ^= 1u << buf;
            const CallBuf& B = W.buf[buf];
            const int lane_cells = (int)N - (int)(c * kCChunk) - lane * 16;
            if (lane_cells > 0) {
                const uint4 vb = *reinterpret_cast<const uint4*>(B.base + lane * 16);
                const uint32_t wb[4] = {vb.x, vb.y, vb.z, vb.w};
                const int n = lane_cells < 16 ? lane_cells : 16;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    if (j < n) {
                        const uint32_t b = (wb[j >> 2] >> (8 * (j & 3))) & 0xffu;
                        const uint32_t cls = call_class(b, ref_code, alt_mask);
                        if (cls < 2u) {
                            const int i = lane * 16 + j;
                            const uint32_t mq = B.mapq[i], bq = B.qual[i], rp = B.rpr[i];
                            cnt0 += cls == 0u; cnt1 += cls;
                            atomicAdd(&W.h_mq[cls][mq], 1u);
                            atomicAdd(&W.h_bq[cls][bq], 1u);
                            if (rp < (uint32_t)kRprBins) atomicAdd(&W.h_rp[cls][rp], 1u);
                            mq_lo = min(mq_lo, mq); mq_hi = max(mq_hi, mq);
                            bq_lo = min(bq_lo, bq); bq_hi = max(bq_hi, bq);
                            rp_lo = min(rp_lo, rp); rp_hi = max(rp_hi, rp);
                        }
                    }
                }
            }
            __syncwarp();
        }
        const unsigned long long n1 = __reduce_add_sync(kFull, cnt0), n2 = __reduce_add_sync(kFull, cnt1);
        mq_lo = __reduce_min_sync(kFull, mq_lo); mq_hi = __reduce_max_sync(kFull, mq_hi);
        bq_lo = __reduce_min_sync(kFull, bq_lo); bq_hi = __reduce_max_sync(kFull, bq_hi);
        rp_lo = __reduce_min_sync(kFull, rp_lo); rp_hi = __reduce_max_sync(kFull, rp_hi);
        int out_mq = 10000, out_rp = 10000, out_bq = 10000;   // one class empty: src/basetype.cpp:233-236
        if (n1 + n2 > 0) {
            const unsigned long long s_mq = hist_twice_ranksum(W.h_mq[0], W.h_mq[1], (int)mq_lo, (int)mq_hi);
            const unsigned long long s_bq = hist_twice_ranksum(W.h_bq[0], W.h_bq[1], (int)bq_lo, (int)bq_hi);
            unsigned long long s_rp = hist_twice_ranksum(W.h_rp[0], W.h_rp[1], (int)min(rp_lo, (uint32_t)kRprBins - 1u),
                                                         (int)min(rp_hi, (uint32_t)kRprBins - 1u));
            if (n1 > 0 && n2 > 0) {
                if (rp_hi >= (uint32_t)kRprBins) s_rp = rpr_pairwise(W, R, N, ref_code, alt_mask, phase);
                if (lane == 0) {
                    out_mq = ranksum_phred(s_mq, n1, n2);
                    out_rp = ranksum_phred(s_rp, n1, n2);
                    out_bq = ranksum_phred(s_bq, n1, n2);
                }
            }
        }
        if (lane == 0) {
            bv_call_out o;
            o.site = site; o.mq_rank_sum = out_mq; o.read_pos_rank_sum = out_rp; o.base_q_rank_sum = out_bq;
            *reinterpret_cast<uint4*>(a.calls + k) = *reinterpret_cast<const uint4*>(&o);
        }
        __syncwarp();
    }
}

// =====================================================================================================================
// K9: free-standing rank-sum tests (bv_ranksum_test), ref_vs_alt_ranksumtest (src/basetype.cpp:201-242) for a batch of
// problems.  A problem is a list of (base code, int32 value) entries, a REF character and an ALT mask; its entries are
// classified by call_class as in K5, and the result is ranksum_phred_double of the exact 2 * (REF rank sum) as K5 forms
// it.  One CTA per problem (grid-stride): a 100,000-read call of the C++ mirror is spread over 256 threads.  Pass 1 counts
// the classes and finds the value range R = vmax - vmin + 1 of the classified entries; then one of three exact paths:
//   narrow    R <= kRsBins: one histogram pass over the entries, then hist_twice_ranksum over R bins (warp 0);
//   windows   the range cut into W = ceil(R / kRsBins) windows from the top, one histogram pass per window, the count of
//             values above the window carried to the next: cost ~ W * (n / kRsThreads + kRsBins / 32) thread steps;
//   pairwise  the smaller class, kRsOwn values per thread in registers, against every classified entry, swept through
//             shared memory (rpr_pairwise's sum): cost ~ ceil(min(n1, n2) / (kRsThreads * kRsOwn)) * n thread steps.
// Between windows and pairwise the kernel takes the smaller estimate; the bound of a problem is that minimum.
// =====================================================================================================================
constexpr int kRsThreads = 256;
constexpr int kRsWarps = kRsThreads / 32;
constexpr int kRsBins = 8192;      // histogram bins per class
constexpr int kRsTile = 2048;      // entries per shared tile of the pairwise sweep
constexpr int kRsOwn = 8;          // values of the owned class a thread holds per sweep
constexpr int kRsCtasPerSm = 3;

struct __align__(128) RsCta {
    uint32_t h[2][kRsBins];        // [class][value - window base], all-zero between problems
    int32_t tv[kRsTile];
    uint8_t tc[kRsTile];
    unsigned long long red_cnt[kRsWarps], red_acc[kRsWarps];
    int32_t red_lo[kRsWarps], red_hi[kRsWarps];
};
constexpr size_t kRsSmemBytes = sizeof(RsCta);
static_assert(kRsCtasPerSm * (kRsSmemBytes + 1024) <= 233472, "K9: kRsCtasPerSm CTAs do not fit the shared memory of an SM");

__device__ __forceinline__ unsigned long long rs_block_sum(unsigned long long x, unsigned long long* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(kFull, x, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = x;
    __syncthreads();
    x = 0;
#pragma unroll
    for (int w = 0; w < kRsWarps; ++w) x += red[w];
    return x;
}

__global__ void __launch_bounds__(kRsThreads) bv_ranksum_test_kernel(const uint8_t* __restrict__ bases,
                                                                     const int32_t* __restrict__ values,
                                                                     const uint64_t* __restrict__ start,
                                                                     const uint8_t* __restrict__ ref_base,
                                                                     const uint8_t* __restrict__ alt_mask, uint32_t n,
                                                                     double* __restrict__ out) {
    RsCta& S = *reinterpret_cast<RsCta*>(bv_smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 2 * kRsBins; i += kRsThreads) (&S.h[0][0])[i] = 0;
    __syncthreads();
#pragma unroll 1
    for (uint32_t p = blockIdx.x; p < n; p += gridDim.x) {
        const uint64_t s0 = start[p], s1 = start[p + 1];
        const int ref_code = ref_code_of(ref_base[p]);
        const uint32_t mask = alt_mask[p];
        // pass 1: class counts (n1 low word, n2 high word) and the value range of the classified entries
        unsigned long long cnt = 0;
        int lo = INT_MAX, hi = INT_MIN;
#pragma unroll 1
        for (uint64_t i = s0 + tid; i < s1; i += kRsThreads) {
            const uint32_t c = call_class(bases[i], ref_code, mask);
            if (c < 2u) {
                const int v = values[i];
                cnt += c == 0u ? 1ull : 1ull << 32;
                lo = min(lo, v); hi = max(hi, v);
            }
        }
        lo = __reduce_min_sync(kFull, lo); hi = __reduce_max_sync(kFull, hi);
        if (lane == 0) { S.red_lo[warp] = lo; S.red_hi[warp] = hi; }
        cnt = rs_block_sum(cnt, S.red_cnt);   // (its barrier publishes red_lo / red_hi too)
#pragma unroll
        for (int w = 0; w < kRsWarps; ++w) { lo = min(lo, S.red_lo[w]); hi = max(hi, S.red_hi[w]); }
        const unsigned long long n1 = cnt & 0xffffffffull, n2 = cnt >> 32, nent = s1 - s0;
        unsigned long long twice = 0;   // 2 * REF rank sum: in warp 0 (histogram paths) or every thread (pairwise)
        if (n1 > 0 && n2 > 0) {
            const unsigned long long range = (unsigned long long)((long long)hi - (long long)lo) + 1ull;
            const unsigned long long wins = (range + kRsBins - 1) / kRsBins;
            const unsigned long long sweeps = (min(n1, n2) + kRsThreads * kRsOwn - 1) / (kRsThreads * kRsOwn);
            if (wins == 1 || wins * ((nent + kRsThreads - 1) / kRsThreads + kRsBins / 32) <= sweeps * nent) {
                unsigned long long above = 0;
#pragma unroll 1
                for (long long top = hi; top >= lo; top -= kRsBins) {   // windows [wlo, top], from the largest values down
                    const long long wlo = max((long long)lo, top - (kRsBins - 1));
#pragma unroll 1
                    for (uint64_t i = s0 + tid; i < s1; i += kRsThreads) {
                        const uint32_t c = call_class(bases[i], ref_code, mask);
                        if (c < 2u) {
                            const long long v = values[i];
                            if (v >= wlo && v <= top) atomicAdd(&S.h[c][(uint32_t)(v - wlo)], 1u);
                        }
                    }
                    __syncthreads();
                    if (warp == 0) twice += hist_twice_ranksum(S.h[0], S.h[1], 0, (int)(top - wlo), &above);
                    __syncthreads();
                }
            } else {
                // pairwise: for every entry i of the owned class, 2 * #{j: v_j > v_i} + #{j: v_j == v_i} + 1 over the
                // classified entries j (i included) is twice its rank
                const uint32_t own = n1 <= n2 ? 0u : 1u;
                unsigned long long acc = 0;
                uint64_t cur = s0 + tid;   // this thread's next entry (stride kRsThreads)
#pragma unroll 1
                for (;;) {
                    int va[kRsOwn];
                    int nk = 0;
#pragma unroll
                    for (int k = 0; k < kRsOwn; ++k) {
                        va[k] = 0;
                        while (cur < s1 && call_class(bases[cur], ref_code, mask) != own) cur += kRsThreads;
                        if (cur < s1) { va[k] = values[cur]; cur += kRsThreads; nk = k + 1; }
                    }
                    if (!__syncthreads_or(nk > 0)) break;
                    acc += (unsigned long long)nk;
#pragma unroll 1
                    for (uint64_t t0 = s0; t0 < s1; t0 += kRsTile) {
                        const uint32_t len = (uint32_t)min((uint64_t)kRsTile, s1 - t0);
                        for (uint32_t j = tid; j < len; j += kRsThreads) {
                            S.tc[j] = (uint8_t)call_class(bases[t0 + j], ref_code, mask);
                            S.tv[j] = values[t0 + j];
                        }
                        __syncthreads();
                        uint32_t a32 = 0;   // <= 2 * kRsTile * kRsOwn
#pragma unroll 1
                        for (uint32_t j = 0; j < len; ++j) {
                            if (S.tc[j] > 1u) continue;   // the same j for every thread
                            const int vj = S.tv[j];
#pragma unroll
                            for (int k = 0; k < kRsOwn; ++k)
                                if (k < nk) a32 += vj > va[k] ? 2u : (vj == va[k] ? 1u : 0u);
                        }
                        acc += a32;
                        __syncthreads();
                    }
                }
                acc = rs_block_sum(acc, S.red_acc);
                const unsigned long long nn = n1 + n2;
                twice = own == 0u ? acc : nn * (nn + 1ull) - acc;   // the ranks 1..nn sum to nn (nn + 1) / 2
            }
        }
        if (tid == 0) out[p] = n1 > 0 && n2 > 0 ? ranksum_phred_double(twice, n1, n2) : 10000.0;   // src/basetype.cpp:233-236
        __syncthreads();
    }
}

// =====================================================================================================================
// K6: population groups.  Shared memory layout and device code of K4 (QualCta / QualWarp, histogram, EM, LRT).
// =====================================================================================================================
__device__ __noinline__ void group_unit(uint32_t k, uint32_t g) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const int lane = threadIdx.x & 31;
    const uint32_t site = cs.a.list_called[k];
    const uint32_t* rec = reinterpret_cast<const uint32_t*>(cs.a.out + site);
    const uint32_t w_alt = rec[kWAlt], w_info = rec[kWInfo];
    const uint32_t n_alt_site = w_alt & 0xffu;
    const int ref_code = ref_code_of(cs.a.ref_base[site]);
    // basecombination = [upper REF, ALT...] (src/basetype_caller.cpp:750-753).  A REF that is not A/C/G/T has no depth
    // entry and is never active (std::map::operator[] gives 0, src/basetype.cpp:137), so it is left out.
    uint32_t order = 0, cand = 0;
    int n_cand = 0;
    if (ref_code >= 0) { order |= (uint32_t)ref_code << (2 * n_cand); cand |= 1u << ref_code; ++n_cand; }
    for (uint32_t i = 0; i < n_alt_site && i < 4u; ++i) {
        const uint32_t b = (i < 3u ? (w_alt >> (8 * (i + 1))) : w_info) & 3u;
        if (cand >> b & 1u) continue;
        order |= b << (2 * n_cand); cand |= 1u << b; ++n_cand;
    }
    // positions past n_cand: the remaining bases (never active, they only complete the permutation)
    for (uint32_t b = 0, p = (uint32_t)n_cand; b < 4u; ++b)
        if (!(cand >> b & 1u)) { order |= b << (2 * p); ++p; }
    if (lane == 0) W.flag_word = 0;
    __syncwarp();

    // BaseType ctor over the group's samples (src/basetype.cpp:22-72): histogram, then depths from it
    const uint32_t h = build_hist(site, cs.a.sample_group, g);
    const uint32_t qmin = h & 0xffu, qmax = (h >> 8) & 0xffu;
    uint32_t dep[5] = {0, 0, 0, 0, 0};
    if (qmin <= qmax) {
#pragma unroll 1
        for (uint32_t q = qmin + lane; q <= qmax; q += 32) {
#pragma unroll
            for (int b = 0; b < 5; ++b) dep[b] += W.hist[b * kQSlots + q];
        }
    }
#pragma unroll
    for (int b = 0; b < 5; ++b) dep[b] = __reduce_add_sync(kFull, dep[b]);
    const uint32_t total = dep[0] + dep[1] + dep[2] + dep[3] + dep[4];
    const double dtot = (double)total;
    __syncwarp();
    if (lane == 0) {
        W.rec.depth[0] = dep[0]; W.rec.depth[1] = dep[1]; W.rec.depth[2] = dep[2]; W.rec.depth[3] = dep[3];
        W.rec.depth_other = dep[4];
        W.flag_word |= h >> 16;
    }
    __syncwarp();

    uint32_t act = 0;
    if (total > 0) {   // src/basetype.cpp:132 returns at once for an uncovered group
        for (int b = 0; b < 4; ++b)
            if ((cand >> b & 1u) && is_active(dep[b], total, dtot, cs.a.min_af)) act |= 1u << b;
    }
    int n_act = __popc(act);
    if (n_act >= 2) {
        const uint32_t r = lrt_multi(qmin, qmax, act, order);
        act = r & 0xfu; n_act = (int)((r >> 4) & 0xfu);
    } else {
        if (n_act == 1) {   // closed form of the single-allele EM, as in K4
            const int b = __ffs(act) - 1;
            const bool bad = qmin == 0 && W.hist[b * kQSlots] != 0;
            const double v = bad ? __longlong_as_double(0x7ff8000000000000ll) : 1.0;
            __syncwarp();
            if (lane < 4) W.res_f[lane] = lane == b ? v : 0.0;
        }
        if (qmin <= qmax) {   // histogram back to zero
#pragma unroll 1
            for (uint32_t q = qmin + lane; q <= qmax; q += 32) {
#pragma unroll
                for (int r = 0; r < 5; ++r) W.hist[r * kQSlots + q] = 0;
            }
        }
    }
    __syncwarp();
    if (lane == 0) {
        bv_group_out o;
        o.n_alt = 0; o.alt[0] = o.alt[1] = o.alt[2] = o.alt[3] = 0; o.flags = (uint8_t)W.flag_word;
        o.reserved[0] = o.reserved[1] = 0;
        o.af[0] = o.af[1] = o.af[2] = o.af[3] = 0.0;
        // ALT = active bases, in list order, that differ from REF (src/basetype.cpp:170-177)
        for (int p = 0; p < n_cand; ++p) {
            const uint32_t b = (order >> (2 * p)) & 3u;
            if ((act >> b & 1u) && (int)b != ref_code) {
                o.alt[o.n_alt] = (uint8_t)b;
                o.af[o.n_alt] = W.res_f[b];
                ++o.n_alt;
            }
        }
        cs.a.groups[(size_t)k * cs.a.n_groups + g] = o;
    }
    __syncwarp();
}

__global__ void __launch_bounds__(kQualWarps * 32, 1) bv_group_kernel(const __grid_constant__ SiteKernelArgs a) {
    QualCta& cs = cta_shared();
    QualWarp& W = warp_smem();
    const int lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < 4 * kQStride; i += blockDim.x) cs.lut[i] = a.lut[i];
    if (threadIdx.x == 0) cs.a = a;
    for (int i = lane; i < kHistWords; i += 32) W.hist[i] = 0;
    if (lane == 0) {
        W.flag_word = 0;
        W.p2_phase = 0;
        for (int b = 0; b < kP2Bufs; ++b) mbar_init(&W.p2bar[b], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint32_t n_units = a.counters[kCntCalled] * a.n_groups;
    for (;;) {
        uint32_t u = 0;
        if (lane == 0) u = atomicAdd(a.counters + kCntGroupNext, 1u);
        u = __shfl_sync(kFull, u, 0);
        if (u >= n_units) break;
        group_unit(u / a.n_groups, u % a.n_groups);
    }
}

}  // namespace bv
