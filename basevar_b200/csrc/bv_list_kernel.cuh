// bv_list_kernel.cuh -- K8 bv_list_kernel: BaseType::lrt(specific_bases) over a per-site ORDERED candidate list
// (src/basetype.h:117-118, src/basetype.cpp:130-199), the overload the population-group path calls with [REF, ALT...]
// (src/basetype_caller.cpp:747-760) and any caller may call with its own alleles.
//
// One warp per site with a non-empty list and counted reads, after the standard kernels: the depths and the strand table
// come from the site's finished record, the (base, phred) histogram of the row from build_hist, and the EM / elimination
// from lrt_on_bins with the list as the candidate order -- the code K4a's fallback and K6 run (the list A,C,G,T gives the record's
// ALT / FS; AF / QUAL too, but to the last bit only where K4b's per-task EM did not decide it: DESIGN.md section 8).  QUAL is
// qual_from_chi, FS the code of bv_fs_kernel (fs_from_table).
// Shared memory layout: QualCta / QualWarp of K4 (the histogram is back to all-zero after every site).
#pragma once
#include "bv_finish_kernels.cuh"

namespace bv {

static_assert(sizeof(bv_lrt_out) == 64, "bv_lrt_out layout (include/basevar_b200.h, capi.LRT_OUT_DTYPE)");

// lists[site] as one word, byte k = k-th entry.  Returns the number of entries before the first BV_LIST_END and packs them
// into `order` (two bits each, position 0 in bits 0-1); -1 for a repeated base or a code outside 0..3.
__host__ __device__ __forceinline__ int list_decode(uint32_t w, uint32_t& order) {
    uint32_t seen = 0;
    order = 0;
    for (int k = 0; k < 4; ++k) {
        const uint32_t c = (w >> (8 * k)) & 0xffu;
        if (c == BV_LIST_END) return k;
        if (c > 3u || (seen >> c & 1u)) return -1;
        seen |= 1u << c;
        order |= c << (2 * k);
    }
    return 4;
}

// kPacked: lrt_out is the site's own entry (the packed list of bv_list_packed_kernel), else the tile's array indexed by site.
template <bool kPacked>
__device__ __noinline__ void list_site(uint32_t site, uint32_t w, bv_lrt_out* __restrict__ lrt_out) {
    QualWarp& W = warp_smem();
    const QualCta& cs = cta_shared();
    const int lane = threadIdx.x & 31;
    uint32_t order = 0;
    const int n_list = list_decode(w, order);
    if (lane < 8) reinterpret_cast<uint4*>(&W.rec)[lane] = reinterpret_cast<const uint4*>(cs.a.out + site)[lane];
    __syncwarp();
    const uint32_t dep[4] = {W.rec.depth[0], W.rec.depth[1], W.rec.depth[2], W.rec.depth[3]};
    const uint32_t total = dep[0] + dep[1] + dep[2] + dep[3] + W.rec.depth_other;
    if (n_list <= 0 || total == 0) {   // skipped, or src/basetype.cpp:132 returns at once: all-zero entry
        if (lane < 4) reinterpret_cast<uint4*>(kPacked ? lrt_out : lrt_out + site)[lane] = make_uint4(0u, 0u, 0u, 0u);
        __syncwarp();
        return;
    }
    // candidate order: the list, then the bases it leaves out (never active, they only complete the permutation)
    uint32_t cand = 0;
    for (int p = 0; p < n_list; ++p) cand |= 1u << ((order >> (2 * p)) & 3u);
    for (uint32_t b = 0, p = (uint32_t)n_list; b < 4u; ++b)
        if (!(cand >> b & 1u)) { order |= b << (2 * p); ++p; }
    if (lane == 0) W.flag_word = W.rec.flags & BV_FLAG_BAD_STRAND;
    __syncwarp();

    // BaseType ctor over the whole row (src/basetype.cpp:22-72)
    const uint32_t h = build_hist(site, nullptr, 0);
    const uint32_t qmin = h & 0xffu, qmax = (h >> 8) & 0xffu;
    if (lane == 0) W.flag_word |= h >> 16;
    __syncwarp();

    const double dtot = (double)total;
    uint32_t act = 0;
    for (int b = 0; b < 4; ++b)
        if ((cand >> b & 1u) && is_active(dep[b], total, dtot, cs.a.min_af)) act |= 1u << b;
    int n_act = __popc(act);
    uint32_t em_calls = 0;
    double chi = 0.0;
    if (n_act >= 2) {
        const uint32_t r = lrt_multi(qmin, qmax, act, order);
        act = r & 0xfu; n_act = (int)((r >> 4) & 0xfu); em_calls = r >> 8;
        chi = W.res_chi;
    } else {
        if (n_act == 1) {   // closed form of the single-allele EM, as in K4a
            const int b = __ffs(act) - 1;
            const bool bad = qmin == 0 && W.hist[b * kQSlots] != 0;
            const double v = bad ? __longlong_as_double(0x7ff8000000000000ll) : 1.0;
            __syncwarp();
            if (lane < 4) W.res_f[lane] = lane == b ? v : 0.0;
            em_calls = 1;
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
        const int ref_code = ref_code_of(cs.a.ref_base[site]);
        uint32_t flags = W.flag_word;
        bv_lrt_out o;
        o.n_alt = 0; o.alt[0] = o.alt[1] = o.alt[2] = o.alt[3] = 0;
        o.n_active = (uint8_t)n_act;
        o.em_calls = (uint8_t)(em_calls > 255u ? 255u : em_calls);
        o.af[0] = o.af[1] = o.af[2] = o.af[3] = 0.0;
        o.qual = 0.0; o.chi2 = chi; o.fs = 0.0;
        // ALT = active bases, in list order, that differ from REF (src/basetype.cpp:170-177)
        uint32_t alt_set = 0;
        for (int p = 0; p < 4; ++p) {
            const uint32_t b = (order >> (2 * p)) & 3u;
            if ((act >> b & 1u) && (int)b != ref_code) {
                o.alt[o.n_alt] = (uint8_t)b;
                o.af[o.n_alt] = W.res_f[b];
                alt_set |= 1u << b;
                ++o.n_alt;
            }
        }
        if (o.n_alt) {
            // QUAL (src/basetype.cpp:180-194): the first active base in list order decides the mono-allelic rule
            const int first_act = nth_active(order, act, 0);
            const double r = (double)dep[first_act] / dtot;
            if (n_act == 1 && total > 10 && r > 0.5) { o.qual = 5000.0; flags |= BV_FLAG_MONO_QUAL; }
            else o.qual = qual_from_chi(chi);
            // strand_bias(REF, ALT set) from the record's strand table (src/basetype.cpp:244-295), as bv_fs_kernel
            int rf, rr, vf, vr, af_, ar;
            strand_tables(&W.rec, ref_code, alt_set, rf, rr, vf, vr, af_, ar);
            if ((vf | vr) != 0 && (rf | rr) != 0) o.fs = fs_from_table(cs.a.logfact, rf, rr, vf, vr);
        }
        o.flags = (uint8_t)flags;
        if (kPacked) *lrt_out = o;
        else lrt_out[site] = o;
    }
    __syncwarp();
}

// shared state of K8's CTA: the tile's arguments, the LUT, every warp's histogram at zero, its mbarriers
__device__ __forceinline__ void list_cta_setup(const SiteKernelArgs& a) {
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
}

__global__ void __launch_bounds__(kQualWarps * 32, 1) bv_list_kernel(const __grid_constant__ SiteKernelArgs a,
                                                                     const uint32_t* __restrict__ lists,
                                                                     bv_lrt_out* __restrict__ lrt_out) {
    list_cta_setup(a);
    // every site of the tile, dealt out statically (a site costs one pass over its row; empty lists cost nothing)
    const uint32_t total_warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t site = (threadIdx.x >> 5) * gridDim.x + blockIdx.x; site < a.n_sites; site += total_warps)
        list_site<false>(site, __ldg(lists + site), lrt_out);
}

// K8 over a packed list (compact results of bv_tile_submit_sparse_lists): pairs[k] = {site, list word} of the k-th listed site,
// its entry goes to lrt_out[k].  The same per-site code as bv_list_kernel, so entry k is the bytes bv_list_kernel gives its site.
__global__ void __launch_bounds__(kQualWarps * 32, 1) bv_list_packed_kernel(const __grid_constant__ SiteKernelArgs a,
                                                                            const uint2* __restrict__ pairs, uint32_t n_pairs,
                                                                            bv_lrt_out* __restrict__ lrt_out) {
    list_cta_setup(a);
    const uint32_t total_warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t k = (threadIdx.x >> 5) * gridDim.x + blockIdx.x; k < n_pairs; k += total_warps) {
        const uint2 p = __ldg(pairs + k);
        list_site<true>(p.x, p.y, lrt_out + k);
    }
}

}  // namespace bv
