// bv_fisher_fast.h -- two-sided Fisher exact test in O(log range + tail) instead of O(range).
//
// kt_fisher_exact (htslib/kfunc.c:245-313) walks the hypergeometric pmf from both ends of its support towards the
// observed table: left = sum of pmf(i), i = lo.., up to the first i_L with pmf(i_L) >= 0.99999999 q (that term is added
// too when it is < 1.00000001 q); right likewise from hi downwards; two = min(1, left + right).  Its cost is the width
// of the support, hundreds to thousands of steps (4 divisions each) at the depths of dense or very wide pileups.
//
// The pmf is unimodal, so i_L is the first crossing of 0.99999999 q on the rising flank [lo, min(n11, mode)] and
// i_R the last one on the falling flank [max(n11, mode), hi]: both are found by bisection on directly evaluated
// pmf values (exp of log-factorial differences, the reference's own hypergeo(), kfunc.c:209-212).  The tail sums run
// outwards from the crossings with the pmf's ratio recurrence (the reference's hypergeo_acc, kfunc.c:220-243) and stop
// when a term no longer changes the sum (< 1e-18 of it): what is dropped is below the rounding of the reference's own
// sum.  Decisions against the two thresholds have a slack of 1e-8 relative, five orders of magnitude above the
// difference between direct and incremental pmf values, and exact ties (symmetric tables) fall inside the slack for
// both.  Checked against the reference's algorithm on random tables in tests/cpp/test_fisher_fast.cpp.
//
// Header-only, host + device: LF(k) returns lgamma(k+1) (glibc values: a table on the device), EXP(x) = exp(x).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define BV_FN __host__ __device__ inline
#else
#define BV_FN inline
#endif

namespace bv {

template <class LF>
BV_FN double ff_lbinom(const LF& lf, int n, int k) {   // kfunc.c:197-201
    if (k == 0 || n == k) return 0;
    return lf(n) - lf(k) - lf(n - k);
}

#if defined(__CUDACC__)
// 1 / m to ~1 ulp: the hardware's 20-bit estimate and two Newton steps (the correctly rounded division costs twice as
// many FP64 instructions).  m == 0 gives NaN, where 1.0 / 0 gives inf: the EM posteriors 0 * inf the reference then forms
// (bv_em_kernels.cuh) are NaN as well.
__device__ __forceinline__ double rcp_fast(double m) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(m));
    double e = fma(-m, r, 1.0);
    r = fma(r, e, r);
    e = fma(-m, r, 1.0);
    return fma(r, e, r);
}
#endif

// num / den in the tail recurrences.  On the device: num * rcp_fast(den) (the correctly rounded FP64 division costs six times
// as many instructions and the tails are hundreds of steps long on deep pileups).  The difference, a few ulp per step, is far
// inside the 1e-8 slack of every decision here.
BV_FN double ff_div(double num, double den) {
#if defined(__CUDA_ARCH__)
    return num * rcp_fast(den);
#else
    return num / den;
#endif
}

template <class LF>
BV_FN double ff_lpmf(const LF& lf, int i, int n1_, int n_1, int n) {   // log of the pmf: the argument of kfunc.c:209-212's exp
    return ff_lbinom(lf, n1_, i) + ff_lbinom(lf, n - n1_, n_1 - i) - ff_lbinom(lf, n, n_1);
}
template <class LF, class EXP>
BV_FN double ff_pmf(const LF& lf, const EXP& ex, int i, int n1_, int n_1, int n) {   // kfunc.c:209-212
    return ex(ff_lpmf(lf, i, n1_, n_1, n));
}

// The fast path is used for wide supports only, and not for astronomically small q: below ~1e-250 the reference's
// incremental products run into denormals and its sum loses terms (it can even return 0, i.e. FS = 10000, where the
// true p is 1e-305); parity there needs its own operation sequence, which the callers keep for exactly that case.
constexpr int kFisherNarrowSupport = 24;   // supports up to this wide are walked as the reference does
BV_FN bool fisher_fast_applicable(int lo, int hi, double q) { return hi - lo > kFisherNarrowSupport && q > 1e-250; }

// Two-sided p of the table (n11 n12 / n21 n22); q_in = pmf(n11) already computed by the caller (> 0), lo < hi.
// side: kFisherBoth = the whole test; kFisherLeft / kFisherRight = that tail's sum alone, not clamped -- the two tails share
// nothing, so two threads can take one each (bv_fisher_kernel); their sum, clamped to 1, is the value of the whole test bit for bit.
constexpr int kFisherBoth = -1, kFisherLeft = 0, kFisherRight = 1;
template <class LF, class EXP>
BV_FN double fisher_two_sided_fast(const LF& lf, const EXP& ex, int n11, int n1_, int n_1, int n, int lo, int hi, double q,
                                   int side = kFisherBoth) {
    const double thr_hi = 1.00000001 * q;
    // The bisections compare LOGARITHMS of the pmf with log(0.99999999 q): the same decisions (exp is monotone, and its rounding is
    // eight orders of magnitude below the slack) without an exp per probe -- the exps were a fifth of the test's instructions.
    const double lthr_lo = ff_lpmf(lf, n11, n1_, n_1, n) + -1.00000000500000003e-8;   // log(0.99999999) = -1.000000005e-8
    int64_t m64 = ((int64_t)n1_ + 1) * ((int64_t)n_1 + 1) / ((int64_t)n + 2);
    int mode = (int)(m64 < lo ? lo : m64 > hi ? hi : m64);
    double two = 0.0;
    if (side != kFisherRight) {   // ---- left: first i in [lo, min(n11, mode)] with pmf(i) >= thr_lo (pmf rises there; the end point qualifies)
        int a = lo, b = n11 < mode ? n11 : mode;
        while (a < b) {
            const int mid = a + ((b - a) >> 1);
            if (ff_lpmf(lf, mid, n1_, n_1, n) >= lthr_lo) b = mid; else a = mid + 1;
        }
        const int iL = a;
        const double pL = iL == n11 ? q : ff_pmf(lf, ex, iL, n1_, n_1, n);
        double left = 0.0;
        if (iL > lo) {
            int i = iL - 1;
            double p = ff_pmf(lf, ex, i, n1_, n_1, n);
            for (;;) {
                left += p;
                if (i == lo || p < 1e-18 * left) break;
                // pmf(i-1) = pmf(i) * i * n22(i) / ((n1_-i+1) (n_1-i+1)),  n22(i) = i + n - n1_ - n_1   (kfunc.c:234-236)
                p *= ff_div((double)i * (double)(i + n - n1_ - n_1), (double)(n1_ - i + 1) * (double)(n_1 - i + 1));   // products < 2^53: exact
                --i;
            }
        }
        if (pL < thr_hi) left += pL;
        two += left;
    }
    if (side != kFisherLeft) {   // ---- right: last i in [max(n11, mode), hi] with pmf(i) >= thr_lo (pmf falls there; the start point qualifies)
        int a = n11 > mode ? n11 : mode, b = hi;
        while (a < b) {
            const int mid = a + ((b - a + 1) >> 1);
            if (ff_lpmf(lf, mid, n1_, n_1, n) >= lthr_lo) a = mid; else b = mid - 1;
        }
        const int iR = a;
        const double pR = iR == n11 ? q : ff_pmf(lf, ex, iR, n1_, n_1, n);
        double right = 0.0;
        if (iR < hi) {
            int i = iR + 1;
            double p = ff_pmf(lf, ex, i, n1_, n_1, n);
            for (;;) {
                right += p;
                if (i == hi || p < 1e-18 * right) break;
                // pmf(i+1) = pmf(i) * (n1_-i) (n_1-i) / ((i+1) n22(i+1))                                  (kfunc.c:228-230)
                p *= ff_div((double)(n1_ - i) * (double)(n_1 - i), (double)(i + 1) * (double)(i + 1 + n - n1_ - n_1));
                ++i;
            }
        }
        if (pR < thr_hi) right += pR;
        two += right;
    }
    return (side == kFisherBoth && two > 1.) ? 1. : two;
}

}  // namespace bv
