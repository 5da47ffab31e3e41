// MMSE_CE (`Task 5/MMSE_CE.m:1-39`) for a batch that shares its channel statistics: one power-delay profile h (hence one
// tau_rms, :19-24) and one SNR for all B streams -- the situation of a Monte-Carlo point, `Task5_part2.m:176-177`.
// Then Rpp (:31-35) is ONE Hermitian-Toeplitz matrix and
//     H(1:Np) = Htilde - Rpp^{-1} Htilde / snr = W Htilde,   W = I - Rpp^{-1} / snr      (rows Np+1.. of Rhp are discarded, :38)
// is one Np x Np matrix for the whole batch: it is built once (Np Levinson solves on unit vectors, double) and applied
// to all streams as a complex matrix product on the tensor cores -- tcgen05, TF32 operands with a two-term split of BOTH
// factors (hi*hi + lo*hi + hi*lo concatenated along K, FP32 accumulation in TMEM).  The tensor core's accumulator
// rounds toward zero at every step (measured: a relative bias of ~3e-8 per tcgen05.mma, 2.8e-5 over the 768 steps of
// Np = 1024), so K is cut into slices of 96 steps whose partial products are added in FP32 by the spline kernel:
// ~4e-6 against the float64 oracle.
// The per-stream Levinson kernel (chest.cu) remains the general case (per-stream h / SNR, FP64 contexts).
#include "interp.cuh"
#include "tc_gemm.cuh"

const void* ofdm_upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex);
#define MS_THREADS 128

// c = 2*pi*tau_rms/N_carrier*Nps and snr (linear) from the shared h and SNR_dB: out[0] = c, out[1] = snr
template <typename T>
__global__ void mmse_stats_kernel(const cx<T>* __restrict__ h, int h_len, double Nps, int N_carrier, double snr_db, double* __restrict__ out) {
    __shared__ double red[3][32];
    double v0 = 0, v1 = 0, v2 = 0;
    for (int k = threadIdx.x; k < h_len; k += blockDim.x) {
        const double2 hv = to_d(h[k]);
        const double pw = hv.x * hv.x + hv.y * hv.y;
        v0 += pw; v1 += pw * k; v2 += pw * (double)k * (double)k;
    }
    v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = v0; red[1][threadIdx.x >> 5] = v1; red[2][threadIdx.x >> 5] = v2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, b = 0, c2 = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += red[0][w]; b += red[1][w]; c2 += red[2][w]; }
        const double r = b / a, r2 = c2 / a;
        out[0] = 2.0 * CUDART_PI * sqrt(fmax(r2 - r * r, 0.0)) / (double)N_carrier * Nps;
        out[1] = pow(10.0, snr_db * 0.1);
    }
}

// rows[b][0..n) = src[0..n) for every b: the shared impulse response replicated for the per-stream solver
__global__ void mmse_replicate_kernel(const unsigned char* __restrict__ src, size_t row_bytes, int64_t B, unsigned char* __restrict__ rows,
                                      double* __restrict__ snr, double snr_db) {
    const int64_t b = blockIdx.x;
    for (size_t i = threadIdx.x; i < row_bytes; i += blockDim.x) rows[b * row_bytes + i] = src[i];
    if (threadIdx.x == 0) snr[b] = snr_db;
}

__device__ __forceinline__ void ms_block_sum4(double v[4], double (*red)[4]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = warp_sum(v[q]);
    __syncthreads();
    if (lane == 0) { red[w][0] = v[0]; red[w][1] = v[1]; red[w][2] = v[2]; red[w][3] = v[3]; }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) { double s = 0; for (int k = 0; k < MS_THREADS / 32; ++k) s += red[k][q]; v[q] = s; }
}
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }   // exactly representable in TF32

// Block j: Levinson solve Rpp x = e_j, column j of W = I - Rpp^{-1}/snr, written into the GEMM's B operand
//   Bt [2*Npad rows x 3*K2 columns], row i: Re out, row Npad + i: Im out; K segments [hi | hi | lo], each [Re part | Im part].
__global__ void __launch_bounds__(MS_THREADS) mmse_weight_kernel(const double* __restrict__ stats, int Np, int Npad, int K2, float* __restrict__ Bt) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double red[MS_THREADS / 32][4];
    double2* t = (double2*)smem_raw;
    double2* f = t + Np;
    double2* f2 = f + Np;
    double2* x = f2 + Np;
    const int j = blockIdx.x, tid = threadIdx.x;
    const double c = stats[0], snr = stats[1];
    for (int m = tid; m < Np; m += MS_THREADS) {
        const double den = 1.0 + c * c * (double)m * (double)m;            // 1/(1 + 1j*c*m) = (1 - 1j*c*m)/den   (`MMSE_CE.m:30-35`)
        t[m] = make_double2(1.0 / den + (m == 0 ? 1.0 / snr : 0.0), -c * (double)m / den);
    }
    __syncthreads();
    if (tid == 0) { f[0] = make_double2(1.0 / t[0].x, 0.0); x[0] = j == 0 ? make_double2(1.0 / t[0].x, 0.0) : make_double2(0, 0); }
    __syncthreads();
    double2* fc = f; double2* fn = f2;
    for (int m = 1; m < Np; ++m) {
        double a[4] = {0, 0, 0, 0};
        for (int i = tid; i < m; i += MS_THREADS) {
            const double2 tv = t[m - i];
            const double2 e1 = cmul(tv, fc[i]), e2 = cmul(tv, x[i]);
            a[0] += e1.x; a[1] += e1.y; a[2] += e2.x; a[3] += e2.y;
        }
        ms_block_sum4(a, red);
        const double2 ef = make_double2(a[0], a[1]), ex = make_double2(a[2], a[3]);
        const double den = 1.0 - (ef.x * ef.x + ef.y * ef.y);
        for (int i = tid; i <= m; i += MS_THREADS) {
            const double2 fi = (i < m) ? fc[i] : make_double2(0, 0);
            const double2 bi = (i >= 1) ? cconj(fc[m - i]) : make_double2(0, 0);
            fn[i] = cscale(fi - cmul(ef, bi), 1.0 / den);
        }
        __syncthreads();
        const double2 g = (m == j ? make_double2(1, 0) : make_double2(0, 0)) - ex;
        for (int i = tid; i <= m; i += MS_THREADS) {
            const double2 xi = (i < m) ? x[i] : make_double2(0, 0);
            x[i] = xi + cmul(g, cconj(fn[m - i]));
        }
        double2* tmp = fc; fc = fn; fn = tmp;
        __syncthreads();
    }
    const size_t ld = 3 * (size_t)K2;
    for (int i = tid; i < Np; i += MS_THREADS) {
        const float wr = (float)((i == j ? 1.0 : 0.0) - x[i].x / snr), wi = (float)(-x[i].y / snr);
        const float whr = tf32_hi(wr), whi = tf32_hi(wi);
        float* r0 = Bt + (size_t)i * ld;                 // Re out = sum_j Re W Re Ht - Im W Im Ht
        float* r1 = Bt + (size_t)(Npad + i) * ld;        // Im out = sum_j Im W Re Ht + Re W Im Ht
        r0[j] = whr; r0[Npad + j] = -whi; r0[K2 + j] = whr; r0[K2 + Npad + j] = -whi; r0[2 * K2 + j] = wr - whr; r0[2 * K2 + Npad + j] = -(wi - whi);
        r1[j] = whi; r1[Npad + j] = whr;  r1[K2 + j] = whi; r1[K2 + Npad + j] = whr;  r1[2 * K2 + j] = wi - whi; r1[2 * K2 + Npad + j] = wr - whr;
    }
}

// A operand: row b = [hi(Re Ht, Im Ht) | lo | hi], Ht = Y(pilot_loc, 1) ./ Xp(:, 1)   (`MMSE_CE.m:17`)
__global__ void mmse_ls_split_kernel(const float2* __restrict__ grid, int64_t stream_stride, int64_t B, const int32_t* __restrict__ loc0, int Np, int Npad,
                                     int K2, const float2* __restrict__ xp, float* __restrict__ At) {
    const int64_t b = blockIdx.x;
    float* row = At + b * 3 * (size_t)K2;
    for (int q = threadIdx.x; q < Npad; q += blockDim.x) {
        float2 v = make_float2(0.f, 0.f);
        if (b < B && q < Np) v = cdiv(grid[b * stream_stride + loc0[q]], xp[q]);
        const float hr = tf32_hi(v.x), hi = tf32_hi(v.y);
        row[q] = hr; row[Npad + q] = hi;
        row[K2 + q] = v.x - hr; row[K2 + Npad + q] = v.y - hi;
        row[2 * K2 + q] = hr; row[2 * K2 + Npad + q] = hi;
    }
}

// sum over the K slices of D, row b = [Re H(1:Np) | Im H(1:Np)] -> spline to 1..N_carrier (`MMSE_CE.m:38`)
__global__ void __launch_bounds__(256) mmse_spline_kernel(const float* __restrict__ D, int ldd, int Npad, int n_slices, size_t slice_stride, PlanDev<float> p,
                                                          float2* __restrict__ H) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* y = (float2*)smem_raw;
    float2* d = y + p.n_knots;
    const int64_t b = blockIdx.x;
    const float* row = D + b * (size_t)ldd;
    for (int k = threadIdx.x; k < p.n_src; k += blockDim.x) {
        float re = 0.f, im = 0.f;
        for (int s = 0; s < n_slices; ++s) { re += row[s * slice_stride + k]; im += row[s * slice_stride + Npad + k]; }
        y[p.ext_lo + k] = make_float2(re, im);
    }
    __syncthreads();
    plan_apply(p, y, d, H + b * p.nq);
}

extern "C" int ofdm_mmse_ce_shared(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, const int32_t* loc, int Np, const double* pv, int Nc,
                                   const void* h, int h_len, double snr_db, void* H) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && H && loc && pv && h && Np >= 2 && Nc >= Np && h_len >= 1 && S > 0 && B >= 0, "bad argument");
    if (B == 0) return OFDM_OK;
    const bool tc_ok = ctx->precision == OFDM_PREC_F32 && B >= 256 && Np >= 32 && tc_get_encode() && !getenv("OFDM_B200_NO_TC");
    if (!tc_ok) {
        // general path: replicate the shared statistics and run the per-stream solver
        const size_t esz = ctx->precision == OFDM_PREC_F64 ? sizeof(double2) : sizeof(float2);
        unsigned char* tmp = nullptr;
        const size_t rows_b = (esz * (size_t)h_len * B + 15) / 16 * 16;
        CUDA_TRY(ctx, cudaMallocAsync((void**)&tmp, rows_b + sizeof(double) * B, ctx->stream));
        double* snr_d = (double*)(tmp + rows_b);
        mmse_replicate_kernel<<<(unsigned)B, 64, 0, ctx->stream>>>((const unsigned char*)h, esz * (size_t)h_len, B, tmp, snr_d, snr_db);
        ctx->launches++;
        int rc = ofdm_mmse_ce(ctx, grid, B, S, Nfft, loc, Np, pv, Nc, tmp, h_len, snr_d, H);
        cudaFreeAsync(tmp, ctx->stream);
        return rc;
    }
    std::vector<int32_t> p0(Np);
    for (int i = 0; i < Np; ++i) {
        REQUIRE(ctx, loc[i] >= 1 && loc[i] <= std::min(Nfft, Nc) && (i == 0 || loc[i] > loc[i - 1]), "pilot locations must increase within 1..N_carrier");
        p0[i] = loc[i] - 1;
    }
    const int32_t* l0 = (const int32_t*)ctx_blob(ctx, p0.data(), sizeof(int32_t) * Np);
    const InterpPlan* pl = ctx_plan(ctx, loc, Np, Nc, nullptr, Nc, OFDM_INTERP_SPLINE);
    const void* xp = ofdm_upload_pilots(ctx, pv, Np);
    REQUIRE(ctx, l0 && pl && xp, "plan construction failed");
    const int Npad = (Np + 63) / 64 * 64;                  // 2*Npad is a multiple of the 128-column tile
    const int K2 = 2 * Npad;                               // one K segment: [Re | Im]
    const int64_t Bpad = (B + TC_BM - 1) / TC_BM * TC_BM;
    cudaStream_t st = ctx->stream;
    float *At = nullptr, *Bt = nullptr, *D = nullptr;
    double* stats = nullptr;
    const int Kt = 3 * K2;                                 // whole K of the split product
    const int Ks = 768;                                    // K per slice = 96 tcgen05.mma steps per accumulator
    const int n_slices = (Kt + Ks - 1) / Ks;               // Kt is a multiple of 384; the last slice may be half a slice
    const size_t slice_stride = (size_t)Bpad * 2 * Npad;
    // one stream-ordered allocation for the four temporaries (one failure point, one release)
    const size_t at_b = sizeof(float) * (size_t)Bpad * 3 * K2, bt_b = sizeof(float) * (size_t)2 * Npad * 3 * K2, d_b = sizeof(float) * slice_stride * n_slices;
    unsigned char* pool = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync((void**)&pool, at_b + bt_b + d_b + 64, st));
    At = (float*)pool; Bt = (float*)(pool + at_b); D = (float*)(pool + at_b + bt_b); stats = (double*)(pool + at_b + bt_b + d_b);
    if (cudaMemsetAsync(Bt, 0, bt_b, st) != cudaSuccess) { cudaFreeAsync(pool, st); return ctx_fail(ctx, OFDM_ERR_CUDA, "memset failed"); }
    mmse_stats_kernel<float><<<1, 256, 0, st>>>((const float2*)h, h_len, (double)(loc[1] - loc[0]), Nc, snr_db, stats);
    const size_t wsm = 4 * sizeof(double2) * (size_t)Np;
    int rc = OFDM_OK;
    if (wsm > 48 * 1024) func_smem_optin((const void*)mmse_weight_kernel, (int)wsm);
    mmse_weight_kernel<<<Np, MS_THREADS, wsm, st>>>(stats, Np, Npad, K2, Bt);
    mmse_ls_split_kernel<<<(unsigned)Bpad, 128, 0, st>>>((const float2*)grid, (int64_t)S * Nfft, B, l0, Np, Npad, K2, (const float2*)xp, At);
    if (rc == OFDM_OK) {
        func_smem_optin((const void*)tc_gemm_store_kernel, TC_SMEM_BYTES);
        for (int s = 0; s < n_slices && rc == OFDM_OK; ++s) {
            const int k0 = s * Ks, kn = std::min(Ks, Kt - k0);
            CUtensorMap mapA, mapB;
            if (!tc_make_kmajor_map(&mapA, At + k0, (uint64_t)Bpad, (uint64_t)kn, (uint64_t)Kt) ||
                !tc_make_kmajor_map(&mapB, Bt + k0, (uint64_t)2 * Npad, (uint64_t)kn, (uint64_t)Kt)) {
                rc = ctx_fail(ctx, OFDM_ERR_CUDA, "cuTensorMapEncodeTiled failed");
                break;
            }
            tc_gemm_store_kernel<<<dim3((unsigned)(2 * Npad / TC_BN), (unsigned)(Bpad / TC_BM)), TC_THREADS, TC_SMEM_BYTES, st>>>(mapA, mapB, D + s * slice_stride,
                                                                                                                                2 * Npad, kn, 1);
            ctx->launches++;
        }
    }
    if (rc == OFDM_OK) {
        const size_t ssm = 2 * sizeof(float2) * (size_t)pl->n_knots;
        if (ssm > 48 * 1024) func_smem_optin((const void*)mmse_spline_kernel, (int)ssm);
        mmse_spline_kernel<<<(unsigned)B, 256, ssm, st>>>(D, 2 * Npad, Npad, n_slices, slice_stride, plan_dev<float>(pl), (float2*)H);
        ctx->launches += 4;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "shared-statistics MMSE launch failed: %s", cudaGetErrorString(e));
    }
    cudaFreeAsync(pool, st);
    return rc;
}
