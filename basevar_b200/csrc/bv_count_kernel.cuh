// bv_count_kernel.cuh -- K1: the streaming pass over every cell (see bv_common.cuh for the split of the core into kernels).
//
// One warp owns one genomic site at a time (sites are the embarrassingly parallel axis, samples the reduction axis).
// Persistent CTAs, one per SM; every warp streams its own sequence of site rows (warp w: sites w, w + W, ...) through
// a private ring of TMA-filled shared-memory stages: lane 0 issues cp.async.bulk for the unit kCountStages-1 ahead,
// the stage's mbarrier flips when the bytes have landed (SASS UBLKCP / SYNCS.ARRIVE.TRANS64 / SYNCS.PHASECHK).
//
// Only the base and strand planes are read here.  Per 16-cell vector a lane spends ~50 integer instructions:
// SIMD-in-register byte arithmetic finds the counted cells (code < 5) and the cells equal to REF, dp4a counts them and
// their '-' strands; the (rare) counted cells that are NOT the reference base -- sequencing errors, ALT alleles --
// are counted one by one into ten shared-memory counters.  Result per site: per-base depths and the 2x4 strand table,
// bit-exact (BaseType::BaseType, src/basetype.cpp:45-71; strand_bias counting, src/basetype.cpp:252-274).
//
// A site whose counted cells all equal REF (the common case) has a closed-form record -- one active allele == REF, the
// EM's answer is f = 1, no ALT, QUAL / FS = 0 -- which 32 lanes compose in registers and store coalesced.  Every other
// site gets its counts and goes onto the work list of K2.
#pragma once
#include "bv_common.cuh"

namespace bv {

// Two shapes of the kernel (warps per CTA x ring depth per warp), chosen by the row length at launch.  Measured on
// B200 (profiles/history/r01o_k1_ring_shapes.txt): rows of <= 1,000 samples want many warps (per-site work is short, 32 warps
// keep the issue slots 82 % busy), rows of 10,000 samples want deeper rings on fewer warps (0.66 ms vs 0.93 ms per
// 10^9 cells).
constexpr int kCountWarpsShort = 32, kCountStagesShort = 3;
constexpr int kCountWarpsLong = 16, kCountStagesLong = 4;
constexpr int kLongRowSamples = 4096;         // rows longer than this use the *Long shape
constexpr int kChunk = 1024;                  // cells per stage and plane: two 16-cell vectors per lane
constexpr int kSlowBatch = 16;                // one atomicAdd on the list counter per this many sites

struct __align__(128) Stage {                 // one chunk of the base and strand planes of one site row
    uint8_t base[kChunk];
    uint8_t strand[kChunk];
};

template <int kCountStages>
struct __align__(128) CountWarp {
    Stage stage[kCountStages];
    uint32_t nr_cnt[12];                      // counted cells that are not the reference base, [2*base + strand]
    uint32_t pad_[4];
    uint32_t slow_buf[kSlowBatch];            // sites for K2, appended to the global list one batch at a time
    uint64_t full[kCountStages];
};

template <int kCountWarps, int kCountStages>
constexpr size_t count_smem_bytes() { return (size_t)kCountWarps * sizeof(CountWarp<kCountStages>); }
static_assert(count_smem_bytes<kCountWarpsShort, kCountStagesShort>() <= 232448, "shared memory of the count kernel exceeds 227 KB");
static_assert(count_smem_bytes<kCountWarpsLong, kCountStagesLong>() <= 232448, "shared memory of the count kernel exceeds 227 KB");

struct ScanAcc {
    uint32_t nref;     // 128 * (# cells holding the reference base)
    uint32_t nrev;     // 128 * (# of those on the '-' strand)
    uint32_t nonref;   // != 0: the row has counted cells that are not the reference base
    uint32_t bad;      // != 0: a counted cell has a strand code other than +/-
};

// SIMD-in-register scan of 4 cells (one 32-bit word of the base plane and of the strand plane).  Every mask has its
// information in bit 7 of each byte.  Returns the mask of counted cells that are not the reference base.
__device__ __forceinline__ uint32_t scan_word(uint32_t wb, uint32_t ws, uint32_t refw, ScanAcc& A) {
    // counted: base code < 5 (A,C,G,T,other); bytes >= 0x80 are never counted
    const uint32_t m = ~(((wb | 0x80808080u) - 0x05050505u) | wb) & 0x80808080u;
    // equal to the reference base (refw = code * 0x01010101, or 0x08080808 when REF is not A/C/G/T)
    const uint32_t x = (wb ^ refw) & 0x7f7f7f7fu;
    const uint32_t eq = ~((x + 0x7f7f7f7fu) | wb) & 0x80808080u;
    // strand code >= 2 in a counted cell: the reference throws (src/basetype.cpp:271-273)
    A.bad |= (((ws & 0x7f7f7f7fu) + 0x7e7e7e7eu) | ws) & m;
    A.nref = __dp4a(eq, 0x01010101u, A.nref);
    A.nrev = __dp4a(eq, ws, A.nrev);
    return m & ~eq;
}

template <int kCountWarps, int kCountStages>
__global__ void __launch_bounds__(kCountWarps * 32, 1) bv_count_kernel(const __grid_constant__ SiteKernelArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    CountWarp<kCountStages>& W = reinterpret_cast<CountWarp<kCountStages>*>(bv_smem_raw)[warp];

    if (lane < 12) W.nr_cnt[lane] = 0;
    if (lane == 0) {
        for (int s = 0; s < kCountStages; ++s) mbar_init(&W.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    const uint32_t N = a.n_samples, n_sites = a.n_sites;
    const uint32_t total_warps = gridDim.x * kCountWarps;
    const uint32_t warp_global = blockIdx.x * kCountWarps + warp;
    if (warp_global >= n_sites) return;
    const uint32_t row_bytes = (N + 15u) & ~15u;   // bytes of a row that hold cells
    const uint64_t pitch = a.pitch;
    uint32_t* const g_out = reinterpret_cast<uint32_t*>(a.out);
    const uint32_t one_active = (1.0 >= a.min_af) ? 1u : 0u;   // a site whose reads all agree has that allele active
    const uint32_t one_flags = single_em_flag(1u, 1u, a);       // ... and its EM starts from f = 1
    const uint32_t s_stage0 = smem_u32(&W.stage[0]), s_full0 = smem_u32(&W.full[0]);
    // byte masks of the row's last 16-cell vector when N is not a multiple of 16 (one lane, once per row)
    uint32_t keep[4];
    {
        const int valid = (int)(N & 15u);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int left = valid == 0 ? 4 : valid - 4 * k;
            keep[k] = left >= 4 ? 0xffffffffu : (left <= 0 ? 0u : (0xffffffffu >> (8 * (4 - left))));
        }
    }

    // ---- producer cursor: lane 0 issues the bulk copies of the unit kCountStages-1 ahead of the one being scanned ----
    uint32_t p_site = warp_global, p_off = 0, p_slot = 0;
    auto issue = [&]() {
        if (p_site < n_sites) {
            if (lane == 0) {
                const uint32_t bytes = min((uint32_t)kChunk, row_bytes - p_off);
                const size_t g = (size_t)p_site * pitch + p_off;
                const uint32_t bar = s_full0 + 8u * p_slot, dst = s_stage0 + (uint32_t)sizeof(Stage) * p_slot;
                mbar_expect_tx(bar, 2u * bytes);
                bulk_g2s(dst, a.base + g, bytes, bar);
                bulk_g2s(dst + (uint32_t)kChunk, a.strand + g, bytes, bar);
            }
            p_slot = (p_slot + 1 == kCountStages) ? 0 : p_slot + 1;
            p_off += kChunk;
            if (p_off >= row_bytes) { p_off = 0; p_site += total_warps; }
        }
    };
#pragma unroll
    for (int s = 0; s < kCountStages - 1; ++s) issue();

    uint32_t slow_n = 0;
    auto flush_slow = [&]() {   // warp-uniform
        uint32_t pos = 0;
        if (lane == 0) pos = atomicAdd(a.counters + kCntSlow, slow_n);
        pos = __shfl_sync(kFull, pos, 0);
        if ((uint32_t)lane < slow_n) a.list_slow[pos + lane] = W.slow_buf[lane];
        slow_n = 0;
        __syncwarp();
    };

    uint32_t c_slot = 0, c_par = 0;
    uint32_t ref_raw = a.ref_base[warp_global];
#pragma unroll 1
    for (uint32_t site = warp_global; site < n_sites; site += total_warps) {
        // reference base of this site (fetched one site ahead)
        const uint32_t next_site = site + total_warps;
        const uint32_t ref_next = next_site < n_sites ? (uint32_t)__ldg(a.ref_base + next_site) : 0u;
        const int ref_code = ref_code_of(ref_raw);
        const uint32_t refw = ref_code >= 0 ? (uint32_t)ref_code * 0x01010101u : 0x08080808u;

        ScanAcc A;
        A.nref = 0; A.nrev = 0; A.nonref = 0; A.bad = 0;
#pragma unroll 1
        for (uint32_t c_off = 0; c_off < row_bytes; c_off += kChunk) {
            issue();   // goes into the slot the previous unit used; every lane is past it (__syncwarp below)
            mbar_wait(s_full0 + 8u * c_slot, c_par);
#pragma unroll
            for (int v = 0; v < kChunk / 512; ++v) {
                const int lane_cells = (int)N - (int)c_off - v * 512 - lane * 16;
                if (lane_cells > 0) {
                    const uint8_t* cellp = W.stage[c_slot].base + v * 512 + lane * 16;
                    uint4 vb = *reinterpret_cast<const uint4*>(cellp);
                    const uint4 vs = *reinterpret_cast<const uint4*>(cellp + kChunk);
                    if (lane_cells < 16) {
                        vb.x = (vb.x & keep[0]) | (0x05050505u & ~keep[0]); vb.y = (vb.y & keep[1]) | (0x05050505u & ~keep[1]);
                        vb.z = (vb.z & keep[2]) | (0x05050505u & ~keep[2]); vb.w = (vb.w & keep[3]) | (0x05050505u & ~keep[3]);
                    }
                    const uint32_t nr0 = scan_word(vb.x, vs.x, refw, A);
                    const uint32_t nr1 = scan_word(vb.y, vs.y, refw, A);
                    const uint32_t nr2 = scan_word(vb.z, vs.z, refw, A);
                    const uint32_t nr3 = scan_word(vb.w, vs.w, refw, A);
                    if (nr0 | nr1 | nr2 | nr3) {
                        // counted cells that are not the reference base: one by one
                        uint32_t t = (nr0 >> 7) | (nr1 >> 6) | (nr2 >> 5) | (nr3 >> 4);   // bit (8*byte + word)
                        A.nonref |= t;
                        do {
                            int top;
                            asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(t));
                            t ^= 1u << top;
                            const int cell = ((top & 3) << 2) | (top >> 3);
                            const uint32_t b = cellp[cell];
                            const uint32_t s = cellp[cell + kChunk];
                            atomicAdd(&W.nr_cnt[2u * b + (s & 1u)], 1u);
                        } while (t);
                    }
                }
            }
            __syncwarp();
            if (++c_slot == kCountStages) { c_slot = 0; c_par ^= 1u; }
        }

        // ---- the site's record ----
        const uint32_t fl = __reduce_or_sync(kFull, A.nonref | (A.bad ? 0x80000000u : 0u));
        const uint32_t n_ref = __reduce_add_sync(kFull, A.nref) >> 7;
        const uint32_t n_rev = __reduce_add_sync(kFull, A.nrev) >> 7;
        uint32_t w = 0;
        if (fl == 0) {
            // every counted cell holds the reference base (or nothing is covered): final record
            const uint32_t n_active = (n_ref > 0) ? one_active : 0u;
            if (lane == ref_code) w = n_ref;                          // depth[REF]
            if (lane == ref_code + kWFwd) w = n_ref - n_rev;          // fwd[REF]
            if (lane == ref_code + kWRev) w = n_rev;                  // rev[REF]
            if (lane == kWInfo) w = (n_active << 8) | ((n_active ? one_flags : 0u) << 16) | (n_active << 24);   // n_active | flags | em_calls
        } else {
            // counts only: words 0..13 = depth[4], other, state, fwd[4], rev[4]; flags in word 15
            const uint32_t b = lane < 4 ? lane : lane < kWRev ? lane - kWFwd : lane - kWRev;   // base of this word
            if (lane < 4 || (lane >= kWFwd && lane < kWRev + 4)) {
                const uint32_t cf = W.nr_cnt[2u * b], cr = W.nr_cnt[2u * b + 1u];
                const bool is_ref = (int)b == ref_code;
                const uint32_t f = cf + (is_ref ? n_ref - n_rev : 0u), r = cr + (is_ref ? n_rev : 0u);
                w = lane < 4 ? f + r : lane < kWRev ? f : r;
            }
            if (lane == kWOther) w = W.nr_cnt[8] + W.nr_cnt[9];
            if (lane == kWState) w = kStateScalar;
            if (lane == kWInfo) w = (fl >> 31) ? ((uint32_t)BV_FLAG_BAD_STRAND << 16) : 0u;
            if (lane == 0) W.slow_buf[slow_n] = site;
            ++slow_n;
            __syncwarp();
            if (lane < 12) W.nr_cnt[lane] = 0;
            if (slow_n == kSlowBatch) flush_slow();
        }
        g_out[(size_t)site * 32 + lane] = w;
        // compact transport: the two counts the whole record of such a site follows from; 0xffffffff = needs its full record
        // (a brief carries no flags: a covered site whose record has one -- one_flags, at em_max_iter <= 1 or em_eps <= 0 --
        // travels as a full record)
        if (a.brief != nullptr && lane == 0)
            a.brief[site] = fl == 0 && (n_ref == 0 || one_flags == 0u) ? make_uint2(n_ref, n_rev) : make_uint2(0xffffffffu, 0u);
        ref_raw = ref_next;
    }
    if (slow_n) flush_slow();
}

}  // namespace bv
