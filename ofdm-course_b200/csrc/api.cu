// Context, memory, caches and host-side plan construction of libofdm_b200.
#include <cmath>
#include <cstdarg>
#include <algorithm>
#include <mutex>
#include <utility>

#include "common.cuh"

uint64_t fnv1a(const void* p, size_t n, uint64_t h) {
    const unsigned char* c = (const unsigned char*)p;
    for (size_t i = 0; i < n; ++i) { h ^= c[i]; h *= 1099511628211ull; }
    return h;
}

int ctx_fail(ofdm_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}

// ---------------------------------------------------------------- constellation_func
// `Task 5/constellation_func.m:4-29`, including its numeric normalisation.
ConstTable host_constellation(int id) {
    ConstTable c;
    memset(&c, 0, sizeof c);
    int n = 0;
    switch (id) {
    case OFDM_BPSK: { c.bps = 1; n = 2; double r[2] = {-1, 1}; for (int i = 0; i < 2; ++i) { c.re[i] = r[i]; c.im[i] = 0; } break; }
    case OFDM_QPSK: { c.bps = 2; n = 4; double r[4] = {-1, -1, 1, 1}, q[4] = {-1, 1, -1, 1}; for (int i = 0; i < 4; ++i) { c.re[i] = r[i]; c.im[i] = q[i]; } break; }
    case OFDM_8PSK: { c.bps = 3; n = 8; int g[8] = {5, 4, 2, 3, 6, 7, 1, 0}; for (int i = 0; i < 8; ++i) { double a = g[i] * 2 * M_PI / 8; c.re[i] = cos(a); c.im[i] = sin(a); } break; }
    case OFDM_16QAM: {
        c.bps = 4; n = 16;
        double r[16] = {-3, -3, -3, -3, -1, -1, -1, -1, 3, 3, 3, 3, 1, 1, 1, 1};
        double q[16] = {3, 1, -3, -1, 3, 1, -3, -1, 3, 1, -3, -1, 3, 1, -3, -1};
        for (int i = 0; i < 16; ++i) { c.re[i] = r[i]; c.im[i] = q[i]; }
        break; }
    default: c.bps = 0; return c;
    }
    double s = 0;
    for (int i = 0; i < n; ++i) s += c.re[i] * c.re[i] + c.im[i] * c.im[i];
    double norm = sqrt(s / n);
    for (int i = 0; i < n; ++i) { c.re[i] /= norm; c.im[i] /= norm; }
    return c;
}

extern "C" int ofdm_constellation(int constellation, double* table_host, int* bps) {
    ConstTable c = host_constellation(constellation);
    if (c.bps == 0) return OFDM_ERR_INVALID;
    if (bps) *bps = c.bps;
    if (table_host) for (int i = 0; i < (1 << c.bps); ++i) { table_host[2 * i] = c.re[i]; table_host[2 * i + 1] = c.im[i]; }
    return OFDM_OK;
}

extern "C" const char* ofdm_version(void) { return "ofdm_b200 0.1 (sm_100a)"; }

// ---------------------------------------------------------------- context
extern "C" int ofdm_ctx_create(ofdm_ctx** out, int device, int precision) {
    if (!out) return OFDM_ERR_INVALID;
    *out = nullptr;
    if (precision != OFDM_PREC_F32 && precision != OFDM_PREC_F64) return OFDM_ERR_INVALID;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return OFDM_ERR_NODEVICE;  // no CPU fallback by design
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return OFDM_ERR_NODEVICE;
    if (prop.major != 10) return OFDM_ERR_NODEVICE;  // kernels are built for sm_100a only
    if (cudaSetDevice(device) != cudaSuccess) return OFDM_ERR_CUDA;
    ofdm_ctx* ctx = new ofdm_ctx();
    ctx->device = device;
    ctx->precision = precision;
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return OFDM_ERR_CUDA; }
    {   // Stream-ordered temporaries (cudaMallocAsync in the fused chains) are multi-GB: keep freed blocks in the pool
        // instead of returning them to the driver at every synchronisation (the default release threshold is 0).
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = ~(uint64_t)0;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
    }
    ctx->own_stream = true;
    for (int i = 0; i < 2; ++i) cudaStreamCreateWithFlags(&ctx->copy_stream[i], cudaStreamNonBlocking);
    for (int i = 0; i < 4; ++i) cudaEventCreateWithFlags(&ctx->ev[i], cudaEventDisableTiming);
    *out = ctx;
    return OFDM_OK;
}

extern "C" void ofdm_ctx_destroy(ofdm_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto& kv : ctx->blob_cache) cudaFree(kv.second.dev);
    for (auto& kv : ctx->blob_retired) cudaFree(kv.second.dev);
    for (auto& kv : ctx->twiddle_cache) cudaFree(kv.second);
    for (auto& kv : ctx->plan_cache) { cudaFree(kv.second.band); cudaFree(kv.second.qw); cudaFree(kv.second.qk); }
    for (auto& kv : ctx->plan_retired) { cudaFree(kv.second.band); cudaFree(kv.second.qw); cudaFree(kv.second.qk); }
    for (void* p : ctx->owned) cudaFree(p);
    if (ctx->scratch) cudaFree(ctx->scratch);
    for (int i = 0; i < 2; ++i) { if (ctx->staging[i]) cudaFree(ctx->staging[i]); if (ctx->copy_stream[i]) cudaStreamDestroy(ctx->copy_stream[i]); }
    for (int i = 0; i < 4; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* ofdm_last_error(const ofdm_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
extern "C" int ofdm_precision(const ofdm_ctx* ctx) { return ctx ? ctx->precision : OFDM_ERR_INVALID; }
extern "C" int64_t ofdm_launch_count(const ofdm_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int ofdm_ctx_set_stream(ofdm_ctx* ctx, void* s) {
    if (!ctx) return OFDM_ERR_INVALID;
    if (ctx->own_stream && ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); ctx->own_stream = false; }
    if (s) { ctx->stream = (cudaStream_t)s; ctx->own_stream = false; }
    else {
        CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    return OFDM_OK;
}
extern "C" int ofdm_sync(ofdm_ctx* ctx) {
    if (!ctx) return OFDM_ERR_INVALID;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return OFDM_OK;
}
extern "C" int ofdm_malloc(ofdm_ctx* ctx, void** dev, size_t bytes) {
    if (!ctx || !dev) return OFDM_ERR_INVALID;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMalloc(dev, bytes ? bytes : 1));
    return OFDM_OK;
}
extern "C" int ofdm_free(ofdm_ctx* ctx, void* dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    CUDA_TRY(ctx, cudaFree(dev));
    return OFDM_OK;
}
extern "C" int ofdm_memset(ofdm_ctx* ctx, void* dev, int value, size_t bytes) {
    if (!ctx) return OFDM_ERR_INVALID;
    CUDA_TRY(ctx, cudaMemsetAsync(dev, value, bytes, ctx->stream));
    return OFDM_OK;
}
extern "C" int ofdm_h2d(ofdm_ctx* ctx, void* dev, const void* host, size_t bytes) {
    if (!ctx) return OFDM_ERR_INVALID;
    CUDA_TRY(ctx, cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return OFDM_OK;
}
extern "C" int ofdm_d2h(ofdm_ctx* ctx, void* host, const void* dev, size_t bytes) {
    if (!ctx) return OFDM_ERR_INVALID;
    CUDA_TRY(ctx, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return OFDM_OK;
}
extern "C" int ofdm_host_alloc(void** host, size_t bytes) {
    return cudaMallocHost(host, bytes ? bytes : 1) == cudaSuccess ? OFDM_OK : OFDM_ERR_CUDA;
}
extern "C" int ofdm_host_free(void* host) { return cudaFreeHost(host) == cudaSuccess ? OFDM_OK : OFDM_ERR_CUDA; }

cudaError_t func_smem_optin(const void* func, int bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, int> limit;   // (device, kernel) -> limit set so far
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    const auto key = std::make_pair(dev, func);
    const auto it = limit.find(key);
    if (it != limit.end() && it->second >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) limit[key] = bytes;
    return e;
}

// ---------------------------------------------------------------- caches
// Table uploads come from pageable host memory.  cudaMemcpy may return once the data sits in the driver's staging buffer,
// i.e. before the DMA lands, and the kernels that read the tables run on cudaStreamNonBlocking streams that are not
// ordered against the legacy stream -- so every upload is followed by a synchronisation of the legacy stream (a one-time
// cost per cached table).
cudaError_t ctx_upload(void* dev, const void* host, size_t bytes) {
    cudaError_t e = cudaMemcpy(dev, host, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(cudaStreamLegacy);
}

// Cached upload of a small host blob, keyed by a 64-bit content hash and confirmed by the size and a second,
// independent hash (a mismatch probes the next key).  The cache is bounded in two generations: when the live map
// overflows it becomes the retired generation and the PREVIOUS retired generation is freed, so a pointer handed out
// earlier in the same API call (calls take a handful of blobs in sequence) is never freed under the caller.
void* ctx_blob(ofdm_ctx* ctx, const void* host, size_t bytes) {
    uint64_t key = fnv1a(host, bytes) ^ (uint64_t)bytes * 0x9E3779B97F4A7C15ull;
    const uint64_t check = fnv1a(host, bytes, 0x84222325CBF29CE4ull);
    for (int probe = 0; probe < 8; ++probe, ++key) {
        auto it = ctx->blob_cache.find(key);
        if (it == ctx->blob_cache.end()) {
            auto rt = ctx->blob_retired.find(key);
            if (rt == ctx->blob_retired.end()) break;                      // free key: upload below
            if (rt->second.bytes == bytes && rt->second.check == check) {  // still alive in the retired generation
                ctx->blob_cache[key] = rt->second;
                void* d = rt->second.dev;
                ctx->blob_retired.erase(rt);
                return d;
            }
            continue;
        }
        if (it->second.bytes == bytes && it->second.check == check) return it->second.dev;
    }
    if (ctx->blob_cache.size() >= OFDM_BLOB_CACHE_LIMIT) {
        for (auto& kv : ctx->blob_retired) cudaFree(kv.second.dev);       // cudaFree waits for kernels still reading them
        ctx->blob_retired.clear();
        ctx->blob_retired.swap(ctx->blob_cache);
    }
    void* d = nullptr;
    if (cudaMalloc(&d, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    if (ctx_upload(d, host, bytes) != cudaSuccess) { cudaFree(d); return nullptr; }
    ctx->blob_cache[key] = BlobEntry{d, bytes, check};
    return d;
}

void* ctx_scratch(ofdm_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->scratch_bytes) return ctx->scratch;
    if (ctx->scratch) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->scratch); ctx->scratch = nullptr; ctx->scratch_bytes = 0; }
    size_t want = bytes + bytes / 4 + 4096;
    if (cudaMalloc(&ctx->scratch, want) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    ctx->scratch_bytes = want;
    return ctx->scratch;
}

const void* ctx_twiddles(ofdm_ctx* ctx, int N) { return ctx_twiddles_prec(ctx, N, ctx->precision); }

const void* ctx_twiddles_prec(ofdm_ctx* ctx, int N, int precision) {
    uint64_t key = ((uint64_t)N << 1) | (uint64_t)precision;
    auto it = ctx->twiddle_cache.find(key);
    if (it != ctx->twiddle_cache.end()) return it->second;
    void* d = nullptr;
    if (precision == OFDM_PREC_F64) {
        std::vector<double2> t(N);
        for (int k = 0; k < N; ++k) { long double a = -2.0L * M_PIl * k / N; t[k] = make_double2((double)cosl(a), (double)sinl(a)); }
        if (cudaMalloc(&d, sizeof(double2) * N) != cudaSuccess) return nullptr;
        if (ctx_upload(d, t.data(), sizeof(double2) * N) != cudaSuccess) { cudaFree(d); return nullptr; }
    } else {
        std::vector<float2> t(N);
        for (int k = 0; k < N; ++k) { long double a = -2.0L * M_PIl * k / N; t[k] = make_float2((float)cosl(a), (float)sinl(a)); }
        if (cudaMalloc(&d, sizeof(float2) * N) != cudaSuccess) return nullptr;
        if (ctx_upload(d, t.data(), sizeof(float2) * N) != cudaSuccess) { cudaFree(d); return nullptr; }
    }
    ctx->twiddle_cache[key] = d;
    return d;
}

// ---------------------------------------------------------------- interpolation plans
// MATLAB interp1(x, y, xq, 'spline') is the not-a-knot cubic spline (2 knots: line, 3: parabola).
// For a fixed knot set it is a fixed real linear operator on the knot values, which this plan
// tabulates in double on the host: d = D*y (first derivatives at the knots, banded after
// thresholding) and four Hermite weights per query point.
static void solve_tridiag(std::vector<long double>& sub, std::vector<long double>& diag, std::vector<long double>& sup,
                          std::vector<long double>& rhs) {
    const int n = (int)diag.size();
    for (int i = 1; i < n; ++i) {
        long double m = sub[i] / diag[i - 1];
        diag[i] -= m * sup[i - 1];
        rhs[i] -= m * rhs[i - 1];
    }
    rhs[n - 1] /= diag[n - 1];
    for (int i = n - 2; i >= 0; --i) rhs[i] = (rhs[i] - sup[i] * rhs[i + 1]) / diag[i];
}

// derivative response to the unit vector e_j
static void spline_deriv_column(const std::vector<double>& x, int j, std::vector<long double>& out) {
    const int n = (int)x.size();
    out.assign(n, 0.0L);
    std::vector<long double> dx(n - 1), slope(n - 1, 0.0L);
    for (int i = 0; i < n - 1; ++i) dx[i] = (long double)x[i + 1] - x[i];
    if (j >= 1) slope[j - 1] = 1.0L / dx[j - 1];
    if (j <= n - 2) slope[j] = -1.0L / dx[j];
    if (n == 2) { out[0] = out[1] = slope[0]; return; }
    if (n == 3) {  // parabola through three points
        long double A[3][4] = {{1, 1, 0, 2 * slope[0]},
                               {dx[1], 2 * (dx[0] + dx[1]), dx[0], 3 * (dx[0] * slope[1] + dx[1] * slope[0])},
                               {0, 1, 1, 2 * slope[1]}};
        for (int c = 0; c < 3; ++c) {
            int p = c;
            for (int r = c + 1; r < 3; ++r) if (fabsl(A[r][c]) > fabsl(A[p][c])) p = r;
            for (int k = 0; k < 4; ++k) std::swap(A[c][k], A[p][k]);
            for (int r = 0; r < 3; ++r) if (r != c) { long double m = A[r][c] / A[c][c]; for (int k = c; k < 4; ++k) A[r][k] -= m * A[c][k]; }
        }
        for (int r = 0; r < 3; ++r) out[r] = A[r][3] / A[r][r];
        return;
    }
    std::vector<long double> sub(n, 0.0L), diag(n, 0.0L), sup(n, 0.0L), b(n, 0.0L);
    for (int i = 1; i < n - 1; ++i) {
        sub[i] = dx[i];
        diag[i] = 2 * (dx[i - 1] + dx[i]);
        sup[i] = dx[i - 1];
        b[i] = 3 * (dx[i] * slope[i - 1] + dx[i - 1] * slope[i]);
    }
    long double d0 = (long double)x[2] - x[0];
    diag[0] = dx[1]; sup[0] = d0;
    b[0] = ((dx[0] + 2 * d0) * dx[1] * slope[0] + dx[0] * dx[0] * slope[1]) / d0;
    long double d1 = (long double)x[n - 1] - x[n - 3];
    diag[n - 1] = dx[n - 3]; sub[n - 1] = d1;
    b[n - 1] = (dx[n - 2] * dx[n - 2] * slope[n - 3] + (2 * d1 + dx[n - 2]) * dx[n - 3] * slope[n - 2]) / d1;
    solve_tridiag(sub, diag, sup, b);
    for (int i = 0; i < n; ++i) out[i] = b[i];
}

const InterpPlan* ctx_plan(ofdm_ctx* ctx, const int32_t* knots1, int n, int ext_to, const int32_t* queries1, int nq, int method) {
    uint64_t key = fnv1a(knots1, sizeof(int32_t) * n);
    int hdr[5] = {n, ext_to, nq, method, ctx->precision};
    key = fnv1a(hdr, sizeof hdr, key);
    if (queries1) key = fnv1a(queries1, sizeof(int32_t) * nq, key);
    auto it = ctx->plan_cache.find(key);
    if (it != ctx->plan_cache.end()) return &it->second;
    it = ctx->plan_retired.find(key);
    if (it != ctx->plan_retired.end()) return &it->second;

    InterpPlan p;
    memset(&p, 0, sizeof p);
    p.n_src = n;
    p.nq = nq;
    std::vector<double> x;
    if (ext_to > 0 && knots1[0] > 1) {   // `interpolate.m:7-10`
        p.ext_lo = 1;
        p.lo_den = (double)(knots1[1] - knots1[0]);
        p.lo_mul = (double)(knots1[0] - 1);
        x.push_back(1.0);
    }
    for (int i = 0; i < n; ++i) x.push_back((double)knots1[i]);
    if (ext_to > 0 && knots1[n - 1] < ext_to) {  // `interpolate.m:12-16`
        p.ext_hi = 1;
        p.hi_den = (double)(knots1[n - 1] - knots1[n - 2]);
        p.hi_mul = (double)(ext_to - knots1[n - 1]);
        x.push_back((double)ext_to);
    }
    const int nk = (int)x.size();
    p.n_knots = nk;
    const bool spline = (method == OFDM_INTERP_SPLINE);
    // entries of the derivative operator below tol * max are dropped (they decay like 0.268^distance): 1e-8 is
    // below half an FP32 ulp of the result, 1e-19 below a double's
    const double tol = (ctx->precision == OFDM_PREC_F64) ? 1e-19 : 1e-8;

    // derivative operator, column by column, kept as [lo,hi] ranges above the threshold
    std::vector<std::vector<long double>> cols;
    std::vector<int> clo, chi;
    int hb = 0;
    if (spline) {
        cols.resize(nk); clo.resize(nk); chi.resize(nk);
        long double gmax = 0;
        std::vector<long double> col;
        for (int j = 0; j < nk; ++j) {   // pass 1: global scale (O(n) memory)
            spline_deriv_column(x, j, col);
            for (int i = 0; i < nk; ++i) gmax = std::max(gmax, fabsl(col[i]));
        }
        for (int j = 0; j < nk; ++j) {   // pass 2: trim each column to the entries above tol
            spline_deriv_column(x, j, col);
            int lo = j, hi = j;
            for (int i = 0; i < nk; ++i) if (fabsl(col[i]) > tol * gmax) { lo = std::min(lo, i); hi = std::max(hi, i); }
            clo[j] = lo; chi[j] = hi;
            hb = std::max(hb, std::max(j - lo, hi - j));
            cols[j].assign(col.begin() + lo, col.begin() + hi + 1);
        }
    }
    const bool fold = spline && (p.ext_lo || p.ext_hi) && nk >= 4;
    if (fold) hb = std::max(hb, 2);
    p.hb = hb;
    const int bw = 2 * hb + 1;
    std::vector<double> band((size_t)nk * bw, 0.0);
    if (spline)
        for (int j = 0; j < nk; ++j)
            for (int i = clo[j]; i <= chi[j]; ++i) band[(size_t)(j - i + hb) * nk + i] = (double)cols[j][i - clo[j]];   // tap-major [bw][nk]

    if (fold) {
        // y0 = y1*(1+m) - y2*m with m = (loc1-1)/(loc2-loc1) (`interpolate.m:8-9`), likewise at the far end:
        // substitute into every row so the device operator never touches the two extrapolated knots.
        auto Bm = [&](int i, int j) -> double& { return band[(size_t)(j - i + hb) * nk + i]; };
        if (p.ext_lo) {
            const double m = p.lo_mul / p.lo_den;
            for (int i = 0; i <= std::min(nk - 1, hb); ++i) { double d0 = Bm(i, 0); Bm(i, 1) += d0 * (1 + m); Bm(i, 2) -= d0 * m; Bm(i, 0) = 0; }
        }
        if (p.ext_hi) {
            const double m = p.hi_mul / p.hi_den;
            for (int i = std::max(0, nk - 1 - hb); i < nk; ++i) { double dn = Bm(i, nk - 1); Bm(i, nk - 2) += dn * (1 + m); Bm(i, nk - 3) -= dn * m; Bm(i, nk - 1) = 0; }
        }
        p.folded = 1;
    }
    std::vector<double> qw((size_t)nq * 4);
    std::vector<int32_t> qk(nq);
    for (int q = 0; q < nq; ++q) {
        double xq = queries1 ? (double)queries1[q] : (double)(q + 1);
        int k = (int)(std::upper_bound(x.begin(), x.end(), xq) - x.begin()) - 1;
        k = std::max(0, std::min(k, nk - 2));
        double h = x[k + 1] - x[k];
        double t = (xq - x[k]) / h;
        qk[q] = k;
        if (spline) {
            double t2 = t * t, t3 = t2 * t;
            qw[q] = 2 * t3 - 3 * t2 + 1;
            qw[(size_t)nq + q] = (t3 - 2 * t2 + t) * h;
            qw[(size_t)2 * nq + q] = -2 * t3 + 3 * t2;
            qw[(size_t)3 * nq + q] = (t3 - t2) * h;
        } else {
            qw[q] = 1 - t; qw[(size_t)nq + q] = 0; qw[(size_t)2 * nq + q] = t; qw[(size_t)3 * nq + q] = 0;
        }
    }
    auto upload_real = [&](const std::vector<double>& v) -> void* {
        void* d = nullptr;
        if (ctx->precision == OFDM_PREC_F64) {
            if (cudaMalloc(&d, v.size() * sizeof(double) + 8) != cudaSuccess) return nullptr;
            if (ctx_upload(d, v.data(), v.size() * sizeof(double)) != cudaSuccess) { cudaFree(d); return nullptr; }
        } else {
            std::vector<float> f(v.begin(), v.end());
            if (cudaMalloc(&d, f.size() * sizeof(float) + 8) != cudaSuccess) return nullptr;
            if (ctx_upload(d, f.data(), f.size() * sizeof(float)) != cudaSuccess) { cudaFree(d); return nullptr; }
        }
        return d;
    };
    p.band = upload_real(band);
    p.qw = upload_real(qw);
    if (p.band && p.qw && cudaMalloc((void**)&p.qk, sizeof(int32_t) * nq + 8) != cudaSuccess) p.qk = nullptr;
    if (!p.band || !p.qw || !p.qk || ctx_upload(p.qk, qk.data(), sizeof(int32_t) * nq) != cudaSuccess) {
        cudaFree(p.band); cudaFree(p.qw); cudaFree(p.qk);
        cudaGetLastError();
        return nullptr;
    }
    if (ctx->plan_cache.size() >= OFDM_PLAN_CACHE_LIMIT) {   // two generations, as for the blobs: plans returned earlier in this call stay valid
        for (auto& kv : ctx->plan_retired) { cudaFree(kv.second.band); cudaFree(kv.second.qw); cudaFree(kv.second.qk); }
        ctx->plan_retired.clear();
        ctx->plan_retired.swap(ctx->plan_cache);              // std::map::swap keeps element addresses
    }
    ctx->plan_cache[key] = p;
    return &ctx->plan_cache[key];
}
