// numerics_probe.cu -- TEST ONLY (tests/test_gpu_numerics.py builds it into pytest's temporary directory; it is not part of
// libbasevar_b200.so).  It compiles the library's own source, so every probe kernel calls the shipping device function, and it
// takes its tables from a context of that source (bv_create / upload_tables): the LUT with log_tab's table at d_lut + 4 * kQStride,
// and the glibc log-factorials at d_logfact.
//
// One grid-stride kernel per primitive and one extern "C" wrapper per kernel: host arrays in, host arrays out, synchronous; the
// wrapper returns the CUDA status (0 = cudaSuccess).
#include "../../basevar_b200/csrc/bv_api.cu"

namespace {

constexpr int kProbeThreads = 256;

int probe_blocks(size_t n) {
    const size_t b = (n + kProbeThreads - 1) / kProbeThreads;
    return b < 4096 ? (int)b : 4096;
}

#define PROBE_LOOP(i, n) for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (n); i += (size_t)gridDim.x * blockDim.x)

__global__ void k_log_tab(const double* x, double* y, uint32_t* bad, const double2* tab, size_t n) {
    PROBE_LOOP(i, n) {
        uint32_t b = 0;
        y[i] = bv::log_tab(x[i], tab, b);
        bad[i] = b;
    }
}
__global__ void k_log_ratio(const double* r, double* y, size_t n) { PROBE_LOOP(i, n) y[i] = bv::log_ratio(r[i]); }
__global__ void k_rcp_fast(const double* m, double* y, size_t n) { PROBE_LOOP(i, n) y[i] = bv::rcp_fast(m[i]); }
__global__ void k_ff_div(const double* num, const double* den, double* y, size_t n) { PROBE_LOOP(i, n) y[i] = bv::ff_div(num[i], den[i]); }
__global__ void k_gammaq(const double* s, const double* z, double* y, size_t n) { PROBE_LOOP(i, n) y[i] = bv::gammaq(s[i], z[i]); }
__global__ void k_qual_from_chi(const double* chi, double* y, size_t n) { PROBE_LOOP(i, n) y[i] = bv::qual_from_chi(chi[i]); }
__global__ void k_fisher(const int4* t, int side, const double* lf, double* y, uint8_t* whole, size_t n) {
    PROBE_LOOP(i, n) {
        bool w = false;
        y[i] = bv::fisher_two_sided(lf, t[i].x, t[i].y, t[i].z, t[i].w, side, &w);
        whole[i] = w ? 1 : 0;
    }
}
__global__ void k_fs_from_table(const int4* t, const double* lf, double* y, size_t n) {
    PROBE_LOOP(i, n) y[i] = bv::fs_from_table(lf, t[i].x, t[i].y, t[i].z, t[i].w);
}
__global__ void k_erfc(const double* x, double* y, size_t n) { PROBE_LOOP(i, n) y[i] = bv::erfc_as66(x[i]); }
__global__ void k_ranksum_phred(const unsigned long long* twice, const unsigned long long* n1, const unsigned long long* n2, int* y,
                                size_t n) {
    PROBE_LOOP(i, n) y[i] = bv::ranksum_phred(twice[i], n1[i], n2[i]);
}
__global__ void k_is_active(const uint32_t* dep, const uint32_t* total, double min_af, uint8_t* y, size_t n) {
    PROBE_LOOP(i, n) y[i] = bv::is_active(dep[i], total[i], (double)total[i], min_af) ? 1 : 0;
}
__global__ void k_iabs_trunc(const double* diff, long long* y, size_t n) { PROBE_LOOP(i, n) y[i] = bv::iabs_trunc(diff[i]); }

// Device copies of the wrapper's arrays, freed when the wrapper returns.
struct DevArrays {
    void* ptrs[8] = {};
    int n_ptrs = 0;
    cudaError_t err = cudaSuccess;
    template <class T>
    T* in(const T* host, size_t n) {
        T* d = out<T>(n);
        if (err == cudaSuccess && n) err = cudaMemcpy(d, host, n * sizeof(T), cudaMemcpyHostToDevice);
        return d;
    }
    template <class T>
    T* out(size_t n) {
        void* d = nullptr;
        if (err == cudaSuccess) err = cudaMalloc(&d, (n ? n : 1) * sizeof(T));
        if (d) ptrs[n_ptrs++] = d;
        return static_cast<T*>(d);
    }
    template <class T>
    void back(T* host, const T* dev, size_t n) {
        if (err == cudaSuccess && n) err = cudaMemcpy(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost);
    }
    // after a launch: the launch's own error, then the kernel's (synchronising)
    void launched() {
        if (err == cudaSuccess) err = cudaGetLastError();
        if (err == cudaSuccess) err = cudaDeviceSynchronize();
    }
    ~DevArrays() {
        for (int i = 0; i < n_ptrs; ++i) cudaFree(ptrs[i]);
    }
};

}  // namespace

extern "C" {

int probe_log_tab(bv_ctx* ctx, const double* x, double* y, uint32_t* bad, size_t n) {
    const double2* tab = reinterpret_cast<const double2*>(ctx->d_lut + 4 * bv::kQStride);
    DevArrays d;
    const double* dx = d.in(x, n);
    double* dy = d.out<double>(n);
    uint32_t* db = d.out<uint32_t>(n);
    if (d.err == cudaSuccess && n) { k_log_tab<<<probe_blocks(n), kProbeThreads>>>(dx, dy, db, tab, n); d.launched(); }
    d.back(y, dy, n);
    d.back(bad, db, n);
    return (int)d.err;
}

int probe_log_ratio(const double* r, double* y, size_t n) {
    DevArrays d;
    const double* dr = d.in(r, n);
    double* dy = d.out<double>(n);
    if (d.err == cudaSuccess && n) { k_log_ratio<<<probe_blocks(n), kProbeThreads>>>(dr, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

int probe_rcp_fast(const double* m, double* y, size_t n) {
    DevArrays d;
    const double* dm = d.in(m, n);
    double* dy = d.out<double>(n);
    if (d.err == cudaSuccess && n) { k_rcp_fast<<<probe_blocks(n), kProbeThreads>>>(dm, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

int probe_ff_div(const double* num, const double* den, double* y, size_t n) {
    DevArrays d;
    const double* dn = d.in(num, n);
    const double* dd = d.in(den, n);
    double* dy = d.out<double>(n);
    if (d.err == cudaSuccess && n) { k_ff_div<<<probe_blocks(n), kProbeThreads>>>(dn, dd, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

int probe_gammaq(const double* s, const double* z, double* y, size_t n) {
    DevArrays d;
    const double* ds = d.in(s, n);
    const double* dz = d.in(z, n);
    double* dy = d.out<double>(n);
    if (d.err == cudaSuccess && n) { k_gammaq<<<probe_blocks(n), kProbeThreads>>>(ds, dz, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

int probe_qual_from_chi(const double* chi, double* y, size_t n) {
    DevArrays d;
    const double* dc = d.in(chi, n);
    double* dy = d.out<double>(n);
    if (d.err == cudaSuccess && n) { k_qual_from_chi<<<probe_blocks(n), kProbeThreads>>>(dc, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

// tables: n x {n11, n12, n21, n22}, every total <= max_samples + 1 of ctx; side: bv::kFisherBoth / kFisherLeft / kFisherRight;
// whole[i]: fisher_two_sided's `whole` (the value is the whole test: one possible outcome, or q == 0)
int probe_fisher(bv_ctx* ctx, const int32_t* tables, int side, double* y, uint8_t* whole, size_t n) {
    DevArrays d;
    const int4* dt = reinterpret_cast<const int4*>(d.in(tables, 4 * n));
    double* dy = d.out<double>(n);
    uint8_t* dw = d.out<uint8_t>(n);
    if (d.err == cudaSuccess && n) { k_fisher<<<probe_blocks(n), kProbeThreads>>>(dt, side, ctx->d_logfact, dy, dw, n); d.launched(); }
    d.back(y, dy, n);
    d.back(whole, dw, n);
    return (int)d.err;
}

int probe_fs_from_table(bv_ctx* ctx, const int32_t* tables, double* y, size_t n) {
    DevArrays d;
    const int4* dt = reinterpret_cast<const int4*>(d.in(tables, 4 * n));
    double* dy = d.out<double>(n);
    if (d.err == cudaSuccess && n) { k_fs_from_table<<<probe_blocks(n), kProbeThreads>>>(dt, ctx->d_logfact, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

int probe_erfc(const double* x, double* y, size_t n) {
    DevArrays d;
    const double* dx = d.in(x, n);
    double* dy = d.out<double>(n);
    if (d.err == cudaSuccess && n) { k_erfc<<<probe_blocks(n), kProbeThreads>>>(dx, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

int probe_ranksum_phred(const unsigned long long* twice, const unsigned long long* n1, const unsigned long long* n2, int* y, size_t n) {
    DevArrays d;
    const unsigned long long* dt = d.in(twice, n);
    const unsigned long long* d1 = d.in(n1, n);
    const unsigned long long* d2 = d.in(n2, n);
    int* dy = d.out<int>(n);
    if (d.err == cudaSuccess && n) { k_ranksum_phred<<<probe_blocks(n), kProbeThreads>>>(dt, d1, d2, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

int probe_is_active(const uint32_t* dep, const uint32_t* total, double min_af, uint8_t* y, size_t n) {
    DevArrays d;
    const uint32_t* dd = d.in(dep, n);
    const uint32_t* dt = d.in(total, n);
    uint8_t* dy = d.out<uint8_t>(n);
    if (d.err == cudaSuccess && n) { k_is_active<<<probe_blocks(n), kProbeThreads>>>(dd, dt, min_af, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

int probe_iabs_trunc(const double* diff, long long* y, size_t n) {
    DevArrays d;
    const double* dd = d.in(diff, n);
    long long* dy = d.out<long long>(n);
    if (d.err == cudaSuccess && n) { k_iabs_trunc<<<probe_blocks(n), kProbeThreads>>>(dd, dy, n); d.launched(); }
    d.back(y, dy, n);
    return (int)d.err;
}

}  // extern "C"
