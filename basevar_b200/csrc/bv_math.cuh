// bv_math.cuh -- device-side FP64 numerics of the basetype core (sm_100a).
//
// Every function here restates arithmetic that the reference does on the CPU, in the same
// operation order, so that results differ only by libm-vs-libdevice rounding of log/exp/log10
// (<= 1-2 ulp).  The translation unit is compiled with -fmad=false: the x86-64 reference build
// has no FMA contraction, so a*b+c is two roundings there and must be two roundings here.
//
//   bv_gammaq_half      htslib/kfunc.c:39-52,103-143 (kf_lgamma, _kf_gammap, _kf_gammaq, kf_gammaq)
//   bv_fisher_two_sided htslib/kfunc.c:197-313       (lbinom, hypergeo, hypergeo_acc, kt_fisher_exact)
//   bv_fs_from_table    src/basetype.cpp:277-283     (FS rule of strand_bias)
//   bv_qual_from_chi    src/basetype.cpp:188-194     (QUAL rule of BaseType::lrt)
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "bv_fisher_fast.h"

namespace bv {

// The kernel's hot loop is instruction-cache sensitive (ncu: `no_inst` was the top stall when the kernel was
// ~6600 SASS instructions).  libdevice log/exp/log10 are 40-90 instructions each and get inlined at every call
// site, so the rarely executed numerics (QUAL, Fisher) call them through these out-of-line wrappers.
__device__ __noinline__ double nlog(double x) { return log(x); }
// Below log(DBL_MIN) libdevice's exp returns 0 for x < -745.0 or so, where glibc rounds to the denormal grid down to x = -745.133
// (the smallest denormal): a QUAL of 10000 instead of 3233.07 for chi2 in [1482.25, 1482.51] (tests/test_gpu_numerics.py).  There
// exp(x + 40) * exp(-40) is exact to a few ulp of a normal value, far below the one step of the denormal grid it is rounded to.
__device__ __noinline__ double nexp(double x) {
    return x < -708.39641853226410622 ? exp(x + 40.0) * 4.248354255291589e-18 : exp(x);
}
__device__ __noinline__ double nlog10(double x) { return log10(x); }

// ---- kf_lgamma (AS245), kfunc.c:39-52 ------------------------------------------------------------
__device__ __noinline__ double lgamma_as245(double z) {
    double x = 0;
    x += 0.1659470187408462e-06 / (z + 7);
    x += 0.9934937113930748e-05 / (z + 6);
    x -= 0.1385710331296526 / (z + 5);
    x += 12.50734324009056 / (z + 4);
    x -= 176.6150291498386 / (z + 3);
    x += 771.3234287757674 / (z + 2);
    x -= 1259.139216722289 / (z + 1);
    x += 676.5203681218835 / z;
    x += 0.9999999999995183;
    return nlog(x) - 5.58106146679532777 - z + (z - 0.5) * nlog(z + 6.5);
}

// ---- kf_gammaq(s, z), kfunc.c:103-143 --------------------------------------------------------------
__device__ __noinline__ double gammaq(double s, double z) {
    if (z <= 1. || z < s) {
        double sum = 1.0, x = 1.0;
        for (int k = 1; k < 100; ++k) {
            x *= z / (s + k);
            sum += x;
            if (x / sum < 1e-14) break;
        }
        return 1. - nexp(s * nlog(z) - z - lgamma_as245(s + 1.) + nlog(sum));
    }
    const double tiny = 1e-290;
    double f = 1. + z - s, C = f, D = 0.;
    for (int j = 1; j < 100; ++j) {
        double a = j * (s - j), b = (j << 1) + 1 + z - s, d;
        D = b + a * D;
        if (D < tiny) D = tiny;
        C = b + a / C;
        if (C < tiny) C = tiny;
        D = 1. / D;
        d = C * D;
        f *= d;
        if (fabs(d - 1.) < 1e-14) break;
    }
    return nexp(s * nlog(z) - z - lgamma_as245(s) - nlog(f));
}

// ---- QUAL rule, src/basetype.cpp:188-194 (chi2_test = kf_gammaq(dof/2, chi/2), algorithm.h:44-46) ----
__device__ __noinline__ double qual_from_chi(double chi) {
    double p = gammaq(0.5, chi / 2.0);
    if (isnan(p)) p = 1.0;
    double q = (p != 0.0) ? -10 * nlog10(p) : 10000.0;
    if (q == 0.0) q = 0.0;  // scrubs -0.0
    return q;
}

// ---- Fisher exact test, kfunc.c:197-313 ---------------------------------------------------------------
// logfact[k] = lgamma(k+1) computed on the host with glibc, i.e. the very values the reference's
// lbinom() gets from libm.
struct HgState {
    int n11, n1_, n_1, n;
    double p;
};

__device__ __forceinline__ double lbinom_tab(const double* __restrict__ logfact, int n, int k) {
    if (k == 0 || n == k) return 0;
    return __ldg(logfact + n) - __ldg(logfact + k) - __ldg(logfact + (n - k));
}

struct LogFactTab {   // lgamma(k+1), glibc values tabulated on the host
    const double* lf;
    __device__ __forceinline__ double operator()(int k) const { return __ldg(lf + k); }
};
struct ExpFn {
    __device__ __forceinline__ double operator()(double x) const { return nexp(x); }
};

__device__ __noinline__ double hypergeo_tab(const double* __restrict__ lf, int n11, int n1_, int n_1, int n) {
    return nexp(lbinom_tab(lf, n1_, n11) + lbinom_tab(lf, n - n1_, n_1 - n11) - lbinom_tab(lf, n, n_1));
}

// kfunc.c:220-243 with only n11 moving.  The step's factor a / n11 * b / n22 is formed as (a * b) * (1 / (n11 * n22)) -- integer
// products below 2^53, exact, and a Newton reciprocal (ff_div) -- where the reference divides twice: a few ulp per step, far inside
// the 1e-8 slack of the comparisons the walk feeds, at a third of the instructions.
__device__ __noinline__ double hg_move(const double* __restrict__ lf, HgState& st, int n11) {
    int n22 = n11 + st.n - st.n1_ - st.n_1;
    if ((n11 % 11) && n22) {
        if (n11 == st.n11 + 1) {
            st.p *= ff_div((double)(st.n1_ - st.n11) * (double)(st.n_1 - st.n11), (double)n11 * (double)n22);
            st.n11 = n11;
            return st.p;
        }
        if (n11 == st.n11 - 1) {
            st.p *= ff_div((double)st.n11 * (double)(st.n11 + st.n - st.n1_ - st.n_1), (double)(st.n1_ - n11) * (double)(st.n_1 - n11));
            st.n11 = n11;
            return st.p;
        }
    }
    st.n11 = n11;
    st.p = hypergeo_tab(lf, st.n11, st.n1_, st.n_1, st.n);
    return st.p;
}

// side: see fisher_two_sided_fast -- kFisherBoth returns the test's p; kFisherLeft / kFisherRight return that tail's sum alone
// (not clamped), or the whole answer with `whole` set when the table needs no sums (one possible outcome; q == 0).
__device__ __noinline__ double fisher_two_sided(const double* __restrict__ lf, int n11, int n12, int n21, int n22, int side = kFisherBoth,
                                                bool* whole = nullptr) {
    int n1_ = n11 + n12, n_1 = n11 + n21, n = n11 + n12 + n21 + n22;
    int hi = (n_1 < n1_) ? n_1 : n1_;
    int lo = n1_ + n_1 - n;
    if (lo < 0) lo = 0;
    if (whole) *whole = true;
    if (lo == hi) return 1.;
    HgState st;
    st.n11 = n11; st.n1_ = n1_; st.n_1 = n_1; st.n = n;
    st.p = hypergeo_tab(lf, n11, n1_, n_1, n);
    double q = st.p;
    if (q == 0.0) return 0.0;
    if (whole) *whole = false;
    // wide supports (deep or dense pileups): bisection + short tail sums instead of a walk over the whole support
    if (fisher_fast_applicable(lo, hi, q)) return fisher_two_sided_fast(LogFactTab{lf}, ExpFn{}, n11, n1_, n_1, n, lo, hi, q, side);
    double p, left = 0., right = 0.;
    int i, j;
    if (side != kFisherRight) {
        p = hg_move(lf, st, lo);
        for (i = lo + 1; p < 0.99999999 * q && i <= hi; ++i) {
            left += p;
            p = hg_move(lf, st, i);
        }
        if (p < 1.00000001 * q) left += p;
    }
    if (side != kFisherLeft) {
        // The right walk starts from the observed table again, not from where the left walk stopped (the reference carries its
        // state over, which matters only when the left walk ends next to hi: an incremental step from there instead of a direct
        // evaluation, i.e. the rounding of exp() of lgamma differences, up to ~12 ulp of lgamma(n + 1) relative: 1.3e-10 measured at
        // n = 100,001).  So the two tails share nothing and a lane pair forms the same value as one thread.
        st.n11 = n11; st.p = q;
        p = hg_move(lf, st, hi);
        for (j = hi - 1; p < 0.99999999 * q && j >= 0; --j) {
            right += p;
            p = hg_move(lf, st, j);
        }
        if (p < 1.00000001 * q) right += p;
    }
    double two = left + right;
    if (side == kFisherBoth && two > 1.) two = 1.;
    return two;
}

// A 2x2 table with a margin of 1 has two possible outcomes: the single read of that margin falls into the other
// margin's first or second class, with probabilities k/n and 1 - k/n (k = the observed class's total).  kt_fisher_exact
// (kfunc.c:245-313) then returns the observed probability when it is the smaller of the two and (clamped) 1 otherwise;
// ties are exact (2k == n), far outside its 1e-8 comparison slack.  This is the table of every site with one
// sequencing-error read, the most common reason to need the test at all.
__device__ __forceinline__ bool fisher_margin1(int a, int b, int c, int d, double& p) {
    int k;
    if (c + d == 1) k = c ? a + c : b + d;
    else if (a + b == 1) k = a ? a + c : b + d;
    else if (a + c == 1) k = a ? a + b : c + d;
    else if (b + d == 1) k = b ? a + b : c + d;
    else return false;
    const int n = a + b + c + d;
    p = (2 * k >= n) ? 1.0 : (double)k / (double)n;
    return true;
}

// src/basetype.cpp:277-283
__device__ __forceinline__ double fs_from_p(double p) {
    if (p == 1.0) return 0.0;   // -10*log10(1) = -0.0, scrubbed to +0.0 by the reference's `fs == 0` branch
    double fs = -10 * nlog10(p);
    if (isinf(fs)) fs = 10000;
    else if (fs == 0) fs = 0.0;
    return fs;
}
__device__ __noinline__ double fs_from_table(const double* __restrict__ lf, int rf, int rr, int af, int ar) {
    double p;
    if (!fisher_margin1(rf, rr, af, ar, p)) p = fisher_two_sided(lf, rf, rr, af, ar);
    return fs_from_p(p);
}

// ---- warp reductions ------------------------------------------------------------------------------------
__device__ __noinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One term of EM()'s convergence sum with BV_EM_ABS_INT_TRUNC, (double)abs((int)diff) (src/algorithm.h:245), as the x86-64
// build computes it: cvttsd2si gives INT_MIN for NaN and out-of-range values, and abs(INT_MIN) stays INT_MIN.  The terms are
// integers, so their sum is formed exactly in 64 bits, in any order (the reference's double sum of them is exact too).
__device__ __forceinline__ long long iabs_trunc(double diff) {
    if (!(diff > -2147483649.0 && diff < 2147483648.0)) return -2147483648ll;
    const long long t = (long long)diff;
    return t < 0 ? -t : t;
}

}  // namespace bv
