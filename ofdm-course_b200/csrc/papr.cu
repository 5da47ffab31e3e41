// calculatePAPR / calculate_window_PAPR / calculateCCDF (`Task 5/calculatePAPR.m:2-11`, `calculate_window_PAPR.m:2-15`,
// `calculateCCDF.m:2-6`; Task 2's contribution, called from every later script, `Task 5/Main_model_Task_5.m:89-94`).
// The reference evaluates the windowed PAPR in O(L * Nfft); here a window [i, i+W) that starts in block k of W
// samples is the union of a suffix of block k and a prefix of block k+1, so both the sliding maximum and the sliding
// sum come from one suffix scan and one prefix scan per block (O(L), no subtraction, hence no cancellation).
#include "common.cuh"
#include <type_traits>

#define PAPR_THREADS 256

// ---- calculatePAPR: 10*log10(max|x|^2 / mean|x|^2) per stream
template <typename T>
__global__ void papr_kernel(const cx<T>* __restrict__ x, int64_t L, double* __restrict__ out) {
    __shared__ double red[32];
    const int64_t b = blockIdx.x;
    double peak = 0, sum = 0;
    for (int64_t n = threadIdx.x; n < L; n += blockDim.x) {
        const cx<T> v = x[b * L + n];
        const double p = (double)v.x * (double)v.x + (double)v.y * (double)v.y;
        peak = fmax(peak, p); sum += p;
    }
    sum = block_sum(sum, red);
    // block-wide max through the same scratch
    for (int o = 16; o > 0; o >>= 1) peak = fmax(peak, __shfl_xor_sync(0xffffffffu, peak, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = peak;
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = 0;
        for (int w = 0; w < (int)((blockDim.x + 31) >> 5); ++w) m = fmax(m, red[w]);
        out[b] = 10.0 * log10(m / (sum / (double)L));
    }
}

// One half of the block scan of a window block, shared by window_papr_kernel and papr_stats_kernel so that both sum in
// the same order: half 0 turns ssum / smax[0, W) into suffix (sum, max) scans (runs walk right to left), half 1 turns
// [W, 2W) into prefix scans.  Each thread owns a run of `per` consecutive entries; run totals are combined with a warp
// scan per warp and a serial pass over the warp totals.  Ends with a barrier.
template <typename T>
__device__ __forceinline__ void window_scan_half(double* ssum, T* smax, int W, int per, int half, int tid, int lane, int warp,
                                                 double (*wsum)[PAPR_THREADS / 32], T (*wmax)[PAPR_THREADS / 32]) {
    const int lo = tid * per, hi = min(lo + per, W);
    double s = 0; T m = 0;
    if (half == 0) { for (int j = hi - 1; j >= lo; --j) { s += ssum[j]; m = max(m, smax[j]); ssum[j] = s; smax[j] = m; } }
    else { for (int j = lo; j < hi; ++j) { s += ssum[W + j]; m = max(m, smax[W + j]); ssum[W + j] = s; smax[W + j] = m; } }
    // exclusive combination of the run totals: runs to the right (half 0) / to the left (half 1)
    double es = s; T em = m;
    for (int o = 1; o < 32; o <<= 1) {
        const double ts = half == 0 ? __shfl_down_sync(0xffffffffu, es, o) : __shfl_up_sync(0xffffffffu, es, o);
        const T tm = half == 0 ? __shfl_down_sync(0xffffffffu, em, o) : __shfl_up_sync(0xffffffffu, em, o);
        const bool ok = half == 0 ? (lane + o < 32) : (lane >= o);
        if (ok) { es += ts; em = max(em, tm); }
    }
    const int edge = half == 0 ? 0 : 31;          // lane holding the warp total
    if (lane == edge) { wsum[half][warp] = es; wmax[half][warp] = em; }
    __syncthreads();
    double cs = 0; T cm = 0;                       // totals of the warps further right / left
    if (half == 0) { for (int w = warp + 1; w < PAPR_THREADS / 32; ++w) { cs += wsum[0][w]; cm = max(cm, wmax[0][w]); } }
    else { for (int w = 0; w < warp; ++w) { cs += wsum[1][w]; cm = max(cm, wmax[1][w]); } }
    // carry = (inclusive warp scan - own run) + other warps
    const double carry_s = es - s + cs;
    T carry_m = cm;
    {   // maximum has no inverse: redo the exclusive part from the neighbours' inclusive values
        const T nb = half == 0 ? __shfl_down_sync(0xffffffffu, em, 1) : __shfl_up_sync(0xffffffffu, em, 1);
        const bool ok = half == 0 ? (lane < 31) : (lane > 0);
        if (ok) carry_m = max(carry_m, nb);
    }
    if (half == 0) { for (int j = lo; j < hi; ++j) { ssum[j] += carry_s; smax[j] = max(smax[j], carry_m); } }
    else { for (int j = lo; j < hi; ++j) { ssum[W + j] += carry_s; smax[W + j] = max(smax[W + j], carry_m); } }
    __syncthreads();
}

// ---- calculate_window_PAPR
// One CTA produces the W outputs i = kW .. kW+W-1 of one stream.  Shared memory: power p[0..2W), then in place
// suffix (max, sum) over [0, W) and prefix (max, sum) over [W, 2W) (window_scan_half).
template <typename T>
__global__ void __launch_bounds__(PAPR_THREADS) window_papr_kernel(const cx<T>* __restrict__ x, int64_t L, int W, int64_t n_out, T* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* ssum = (double*)smem_raw;                 // 2W running sums
    T* smax = (T*)(ssum + 2 * (size_t)W);             // 2W running maxima
    __shared__ double wsum[2][PAPR_THREADS / 32];
    __shared__ T wmax[2][PAPR_THREADS / 32];
    const int64_t b = blockIdx.x;
    const int64_t i0 = (int64_t)blockIdx.y * W;
    const cx<T>* r = x + b * L;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int j = tid; j < 2 * W; j += PAPR_THREADS) {
        const int64_t n = i0 + j;
        T p = 0;
        if (n < L) { const cx<T> v = r[n]; p = v.x * v.x + v.y * v.y; }
        ssum[j] = (double)p; smax[j] = p;
    }
    __syncthreads();
    const int per = (W + PAPR_THREADS - 1) / PAPR_THREADS;
    // half 0: suffix scan over [0, W); half 1: prefix scan over [W, 2W)
#pragma unroll
    for (int half = 0; half < 2; ++half) window_scan_half<T>(ssum, smax, W, per, half, tid, lane, warp, wsum, wmax);
    for (int j = tid; j < W; j += PAPR_THREADS) {
        const int64_t i = i0 + j;
        if (i < n_out) {
            double s = ssum[j]; T m = smax[j];
            if (j > 0) { s += ssum[W + j - 1]; m = max(m, smax[W + j - 1]); }
            out[b * n_out + i] = (T)(10.0 * log10((double)m / (s / (double)W)));
        }
    }
}

extern "C" int ofdm_papr(ofdm_ctx* ctx, const void* x, int64_t B, int64_t L, double* papr_db) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, x && papr_db && B >= 0 && L > 0, "bad argument");
    if (B == 0) return OFDM_OK;
    DISPATCH_T(ctx, { papr_kernel<T><<<(unsigned)B, 512, 0, ctx->stream>>>((const cx<T>*)x, L, papr_db); });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_window_papr(ofdm_ctx* ctx, const void* x, int64_t B, int64_t L, int W, void* paprs) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, x && paprs && B >= 0 && W > 0 && L >= W, "bad argument (needs L >= Nfft)");
    REQUIRE(ctx, W <= 8192, "window longer than 8192 samples");
    if (B == 0) return OFDM_OK;
    const int64_t n_out = L - W + 1;
    DISPATCH_T(ctx, {
        const size_t smem = 2 * (size_t)W * (sizeof(double) + sizeof(T));
        auto k = window_papr_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<dim3((unsigned)B, (unsigned)cdiv64(n_out, W)), PAPR_THREADS, smem, ctx->stream>>>((const cx<T>*)x, L, W, n_out, (T*)paprs);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- PAPR statistics of a study (ofdm_sweep_papr, csrc/sweep_papr.cu) without storing a window value
// One CTA walks the window blocks [k0, k1) of one stream (a chunk; a whole stream unless the batch is too small to fill the
// GPU) and so reads data blocks k0 .. k1, each sample once (a chunk re-reads the first block of the next one).  Arithmetic
// and layout are window_papr_kernel's, so every window value is bit-identical to ofdm_window_papr's: block k is
// prefix-scanned in [W, 2W) while the suffix scan of block k-1 waits in [0, W), the windows starting in block k-1 are
// evaluated from both, then block k is suffix-scanned in [0, W).  The samples of block k+1 are loaded into registers at
// the top of iteration k and used at its end.  Every window value v goes to bin min(floor(v / bin_db), n_bins - 1) of a
// shared int32 histogram (negative values from rounding and NaN, an all-zero window, to bin 0), flushed once per CTA into
// the point's int64 row with integer atomics.  max |x|^2 of the stream is combined over chunks as the bit pattern of a
// non-negative double (unsigned max orders those as the values).
__device__ __forceinline__ float window_power(float2 v) { return __fmaf_rn(v.x, v.x, __fmul_rn(v.y, v.y)); }   // as window_papr_kernel's
__device__ __forceinline__ double window_power(double2 v) { return __fma_rn(v.x, v.x, __dmul_rn(v.y, v.y)); }  // contracted p

template <typename T, int PER>
__global__ void __launch_bounds__(PAPR_THREADS) papr_stats_kernel(const cx<T>* __restrict__ x, int64_t L, int W, int64_t n_out, int64_t nbw,
                                                                  int64_t chunk, int chunks, double bin_db, int n_bins,
                                                                  unsigned long long* __restrict__ hist, unsigned long long* __restrict__ peak) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* ssum = (double*)smem_raw;                 // [0, W): suffix scan of the previous block; [W, 2W): prefix scan of this one
    T* smax = (T*)(ssum + 2 * (size_t)W);
    int* h = (int*)(smax + 2 * (size_t)W);            // n_bins counters
    __shared__ double wsum[2][PAPR_THREADS / 32];
    __shared__ T wmax[2][PAPR_THREADS / 32];
    __shared__ double red[PAPR_THREADS / 32];
    const int64_t b = blockIdx.x / chunks;
    const int64_t k0 = (int64_t)(blockIdx.x % chunks) * chunk, k1 = min(k0 + chunk, nbw);
    const cx<T>* r = x + b * L;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (W + PAPR_THREADS - 1) / PAPR_THREADS;
    for (int i = tid; i < n_bins; i += PAPR_THREADS) h[i] = 0;
    cx<T> nx[PER];                                    // samples of the next block, in flight
    T pw[PER];                                        // |x|^2 of this block's samples tid + m * PAPR_THREADS
    double pk = 0;
    auto load = [&](int64_t k) {
#pragma unroll
        for (int m = 0; m < PER; ++m) {
            const int j = tid + m * PAPR_THREADS;
            const int64_t n = k * W + j;
            nx[m] = mk<T>(0, 0);
            if (j < W && n < L) nx[m] = r[n];
        }
    };
    auto power = [&]() {
#pragma unroll
        for (int m = 0; m < PER; ++m) {
            pw[m] = window_power(nx[m]);
            pk = fmax(pk, (double)nx[m].x * (double)nx[m].x + (double)nx[m].y * (double)nx[m].y);   // as papr_kernel
        }
    };
    auto store = [&](int off) {
#pragma unroll
        for (int m = 0; m < PER; ++m) {
            const int j = tid + m * PAPR_THREADS;
            if (j < W) { ssum[off + j] = (double)pw[m]; smax[off + j] = pw[m]; }
        }
    };
    load(k0);
    power();
    for (int64_t k = k0; k <= k1; ++k) {
        if (k < k1) load(k + 1);
        if (k > k0) {
            store(W);
            __syncthreads();
            window_scan_half<T>(ssum, smax, W, per, 1, tid, lane, warp, wsum, wmax);
            // the windows starting in block k-1, a run of consecutive ones per thread: equal bins are counted once per run
            const int lo = tid * per, hi = min(lo + per, W);
            int run_bin = 0, run_n = 0;
            for (int j = lo; j < hi; ++j) {
                if ((k - 1) * W + j >= n_out) break;
                double s = ssum[j]; T m = smax[j];
                if (j > 0) { s += ssum[W + j - 1]; m = max(m, smax[W + j - 1]); }
                const T v = (T)(10.0 * log10((double)m / (s / (double)W)));
                const double q = floor((double)v / bin_db);
                const int bin = q >= (double)(n_bins - 1) ? n_bins - 1 : (q > 0 ? (int)q : 0);
                if (bin != run_bin && run_n) { atomicAdd(&h[run_bin], run_n); run_n = 0; }
                run_bin = bin;
                ++run_n;
            }
            if (run_n) atomicAdd(&h[run_bin], run_n);
            __syncthreads();
        }
        if (k < k1) {
            store(0);
            __syncthreads();
            window_scan_half<T>(ssum, smax, W, per, 0, tid, lane, warp, wsum, wmax);
            power();
        }
    }
    __syncthreads();
    for (int i = tid; i < n_bins; i += PAPR_THREADS) {
        const int c = h[i];
        if (c) atomicAdd(&hist[i], (unsigned long long)c);
    }
    for (int o = 16; o > 0; o >>= 1) pk = fmax(pk, __shfl_xor_sync(0xffffffffu, pk, o));
    if (lane == 0) red[warp] = pk;
    __syncthreads();
    if (tid == 0) {
        double m = 0;
        for (int w = 0; w < PAPR_THREADS / 32; ++w) m = fmax(m, red[w]);
        atomicMax(&peak[b], (unsigned long long)__double_as_longlong(m));
    }
}

// calculatePAPR from the combined maximum and the stream power sum of ofdm_tx_chain_p
__global__ void papr_finish_kernel(const unsigned long long* __restrict__ peak, const double* __restrict__ psum, int64_t B, int64_t L, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) out[i] = 10.0 * log10(__longlong_as_double((long long)peak[i]) / (psum[i] / (double)L));
}

template <typename T> static const void* papr_stats_kernel_for(int W) {
    switch ((W + PAPR_THREADS - 1) / PAPR_THREADS) {
    case 1: return (const void*)papr_stats_kernel<T, 1>;
    case 2: return (const void*)papr_stats_kernel<T, 2>;
    case 4: return (const void*)papr_stats_kernel<T, 4>;
    case 8: return (const void*)papr_stats_kernel<T, 8>;
    case 16: return (const void*)papr_stats_kernel<T, 16>;
    case 32:
        if constexpr (sizeof(T) == 4) return (const void*)papr_stats_kernel<T, 32>;   // FP64 at W = 8192 needs 256 KB of shared memory
        else return nullptr;
    default: return nullptr;
    }
}

static size_t papr_stats_smem(int precision, int W, int n_bins) {
    return 2 * (size_t)W * (sizeof(double) + (precision == OFDM_PREC_F64 ? sizeof(double) : sizeof(float))) + sizeof(int) * (size_t)n_bins;
}

// OFDM_OK when the statistics kernel runs at window length W (a power of two) with n_bins bins on the context's device,
// OFDM_ERR_UNSUPPORTED (with its own message) when its shared memory exceeds the device's opt-in limit per block.
int ofdm_papr_stats_check(ofdm_ctx* ctx, int W, int n_bins, const char* who) {
    const void* k = ctx->precision == OFDM_PREC_F64 ? papr_stats_kernel_for<double>(W) : papr_stats_kernel_for<float>(W);
    const size_t dyn = papr_stats_smem(ctx->precision, W, n_bins);
    int optin = 0;
    CUDA_TRY(ctx, cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    size_t stat = 0;
    if (k) {
        cudaFuncAttributes a;
        CUDA_TRY(ctx, cudaFuncGetAttributes(&a, k));
        stat = a.sharedSizeBytes;
    }
    if (!k || dyn + stat > (size_t)optin)
        return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "%s: the PAPR statistics kernel needs %zu B of shared memory per block at Nfft %d with %d bins in %s, "
                        "above this device's limit of %d B (use fewer bins or an FP32 context)", who, dyn + stat, W, n_bins,
                        ctx->precision == OFDM_PREC_F64 ? "FP64" : "FP32", optin);
    return OFDM_OK;
}

// Histogram (+= into hist, n_bins int64) and per-stream PAPR (papr, B doubles) of B streams of L samples at window length W;
// psum: sum |x|^2 per stream (ofdm_tx_chain_p); peak: B scratch words.  ofdm_papr_stats_check must have passed.
int ofdm_papr_stats(ofdm_ctx* ctx, const void* x, int64_t B, int64_t L, int W, const double* psum, double bin_db, int n_bins, int64_t* hist,
                    double* papr, unsigned long long* peak) {
    const void* k = ctx->precision == OFDM_PREC_F64 ? papr_stats_kernel_for<double>(W) : papr_stats_kernel_for<float>(W);
    REQUIRE(ctx, k != nullptr, "no statistics kernel for this window length");
    const size_t smem = papr_stats_smem(ctx->precision, W, n_bins);
    CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
    int per_sm = 0;
    CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, PAPR_THREADS, smem));
    int64_t n_out = L - W + 1, nbw = cdiv64(n_out, W);
    // two waves of CTAs at least; a chunk spans 8 window blocks or more, so the block it re-reads costs at most 1/8
    int64_t chunks = std::min<int64_t>(std::max<int64_t>(1, cdiv64(2 * (int64_t)std::max(per_sm, 1) * ctx->sm_count, B)), std::max<int64_t>(1, nbw / 8));
    int64_t chunk = cdiv64(nbw, chunks);
    chunks = cdiv64(nbw, chunk);
    REQUIRE(ctx, B * chunks < ((int64_t)1 << 31), "too many streams in one tile");
    CUDA_TRY(ctx, cudaMemsetAsync(peak, 0, sizeof(unsigned long long) * (size_t)B, ctx->stream));
    int ichunks = (int)chunks;
    unsigned long long* h = (unsigned long long*)hist;
    void* args[] = {(void*)&x, &L, &W, &n_out, &nbw, &chunk, &ichunks, &bin_db, &n_bins, &h, &peak};
    CUDA_TRY(ctx, cudaLaunchKernel(k, dim3((unsigned)(B * chunks)), dim3(PAPR_THREADS), args, smem, ctx->stream));
    ctx->launches++;
    papr_finish_kernel<<<(unsigned)cdiv64(B, 256), 256, 0, ctx->stream>>>(peak, psum, B, L, papr);
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- calculateCCDF: [F, x] = ecdf(v); CCDF = 1 - F.  ecdf returns the sorted distinct values with the smallest one
// duplicated in front (F = 0 there).  Sort = bitonic network over a power-of-two copy padded with +inf (the vectors
// are tens of thousands of values: one launch per (k, j) stage, all of them L2-resident), then one CTA walks the
// sorted array and emits (value, 1 - last_rank/n) for the last element of every run of equal values.
template <typename T>
__global__ void bitonic_step_kernel(T* __restrict__ v, int64_t n2, int64_t j, int64_t k) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n2) return;
    const int64_t l = i ^ j;
    if (l > i) {
        const T a = v[i], b = v[l];
        const bool up = (i & k) == 0;
        if ((a > b) == up) { v[i] = b; v[l] = a; }
    }
}
template <typename T>
__global__ void ccdf_pad_kernel(const T* __restrict__ in, int64_t n, int64_t n2, T* __restrict__ v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n2) v[i] = i < n ? in[i] : (T)CUDART_INF;
}
template <typename T>
__global__ void ccdf_emit_kernel(const T* __restrict__ v, int64_t n, T* __restrict__ xs, T* __restrict__ ccdf, int64_t* __restrict__ n_out) {
    __shared__ int wcnt[32];
    __shared__ int64_t base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    if (tid == 0) { base = 1; xs[0] = v[0]; ccdf[0] = (T)1; }      // leading duplicate of the minimum, F = 0
    __syncthreads();
    for (int64_t c0 = 0; c0 < n; c0 += blockDim.x) {
        const int64_t i = c0 + tid;
        const bool last = i < n && (i + 1 == n || v[i + 1] != v[i]);
        const unsigned bal = __ballot_sync(0xffffffffu, last);
        if (lane == 0) wcnt[warp] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < nw; ++w) { if (w < warp) before += wcnt[w]; total += wcnt[w]; }
        if (last) {
            const int64_t o = base + before + __popc(bal & ((1u << lane) - 1u));
            xs[o] = v[i];
            ccdf[o] = (T)(1.0 - (double)(i + 1) / (double)n);
        }
        __syncthreads();
        if (tid == 0) base += total;
        __syncthreads();
    }
    if (tid == 0) *n_out = base;
}

extern "C" int ofdm_ccdf(ofdm_ctx* ctx, const void* values, int64_t n, void* x_out, void* ccdf_out, int64_t* n_out_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, values && x_out && ccdf_out && n_out_dev && n >= 1, "bad argument");
    REQUIRE(ctx, n <= ((int64_t)1 << 26), "more than 2^26 values");
    int64_t n2 = 1;
    while (n2 < n) n2 <<= 1;
    DISPATCH_T(ctx, {
        T* v = (T*)ctx_scratch(ctx, sizeof(T) * (size_t)n2);
        REQUIRE(ctx, v != nullptr, "scratch allocation failed");
        const unsigned grid = (unsigned)cdiv64(n2, 256);
        ccdf_pad_kernel<T><<<grid, 256, 0, ctx->stream>>>((const T*)values, n, n2, v);
        for (int64_t k = 2; k <= n2; k <<= 1)
            for (int64_t j = k >> 1; j > 0; j >>= 1) bitonic_step_kernel<T><<<grid, 256, 0, ctx->stream>>>(v, n2, j, k);
        ccdf_emit_kernel<T><<<1, 1024, 0, ctx->stream>>>(v, n, (T*)x_out, (T*)ccdf_out, n_out_dev);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}
