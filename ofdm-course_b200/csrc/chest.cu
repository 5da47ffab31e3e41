// estimate_channel / LS_CE / MMSE_CE / interpolate / equalize_signal.
#include "interp.cuh"

const void* ofdm_upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex);

static int pilots0(ofdm_ctx* ctx, const int32_t* loc, int Np, int limit, const int32_t** out) {
    std::vector<int32_t> p0(Np);
    for (int i = 0; i < Np; ++i) {
        if (loc[i] < 1 || loc[i] > limit) return ctx_fail(ctx, OFDM_ERR_INVALID, "pilot index %d out of range 1..%d", loc[i], limit);
        if (i && loc[i] <= loc[i - 1]) return ctx_fail(ctx, OFDM_ERR_INVALID, "pilot locations must be strictly increasing");
        p0[i] = loc[i] - 1;
    }
    *out = (const int32_t*)ctx_blob(ctx, p0.data(), sizeof(int32_t) * Np);
    return *out ? OFDM_OK : ctx_fail(ctx, OFDM_ERR_CUDA, "device upload failed");
}

#define CE_THREADS 256

// ---- interpolate (`Task 5/interpolate.m:1-24`)
template <typename T>
__global__ void __launch_bounds__(CE_THREADS) interpolate_kernel(const cx<T>* __restrict__ Hp, PlanDev<T> p, cx<T>* __restrict__ H) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* y = (cx<T>*)smem_raw;
    cx<T>* d = y + p.n_knots;
    const int64_t b = blockIdx.x;
    for (int k = threadIdx.x; k < p.n_src; k += blockDim.x) y[p.ext_lo + k] = Hp[b * p.n_src + k];
    __syncthreads();
    plan_apply(p, y, d, H + b * p.nq);
}

// ---- LS_CE (`Task 5/LS_CE.m:27-31`): LS_est(k) = Y(pilot_loc(k)) ./ Xp(k) -- first symbol only.
template <typename T>
__global__ void __launch_bounds__(CE_THREADS) ls_ce_kernel(const cx<T>* __restrict__ grid, int64_t stream_stride, const int32_t* __restrict__ loc0,
                                                           const cx<T>* __restrict__ Xp, PlanDev<T> p, cx<T>* __restrict__ H) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* y = (cx<T>*)smem_raw;
    cx<T>* d = y + p.n_knots;
    const int64_t b = blockIdx.x;
    const cx<T>* Y = grid + b * stream_stride;
    for (int k = threadIdx.x; k < p.n_src; k += blockDim.x) y[p.ext_lo + k] = cdiv(Y[loc0[k]], Xp[k]);
    __syncthreads();
    plan_apply(p, y, d, H + b * p.nq);
}

// ---- estimate_channel (`Task 5/estimate_channel.m:4-8`): mean over symbols of rx./tx, spline over allCarriers.
template <typename T>
__global__ void __launch_bounds__(CE_THREADS) estimate_channel_kernel(const cx<T>* __restrict__ grid, int S, int Nfft, const int32_t* __restrict__ loc0,
                                                                      const cx<T>* __restrict__ Xp /* Np x S */, PlanDev<T> p, cx<T>* __restrict__ H,
                                                                      cx<T>* __restrict__ Hp_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* y = (cx<T>*)smem_raw;
    cx<T>* d = y + p.n_knots;
    const int64_t b = blockIdx.x;
    const cx<T>* g = grid + b * (int64_t)S * Nfft;
    const int Np = p.n_src;
    for (int k = threadIdx.x; k < Np; k += blockDim.x) {
        T sr = 0, si = 0;
        for (int s = 0; s < S; ++s) { cx<T> q = cdiv(g[(int64_t)s * Nfft + loc0[k]], Xp[(int64_t)s * Np + k]); sr += q.x; si += q.y; }
        cx<T> m = mk<T>(sr / (T)S, si / (T)S);
        y[k] = m;
        if (Hp_out) Hp_out[b * Np + k] = m;
    }
    __syncthreads();
    plan_apply(p, y, d, H + b * p.nq);
}

// ---- MMSE_CE (`Task 5/MMSE_CE.m:13-38`).  Rows 1:Np of Rhp equal Rpp - I/snr, and only those rows
// survive line 38, so H(1:Np) = Ht - Rpp^{-1} Ht / snr: one Hermitian-Toeplitz solve per stream,
// done with Levinson's recursion in double (cond(Rpp) ~ snr*lambda_max is too much for FP32).
// MEAS = true reads the measurement vectors Y = RX(pilot_loc,1)./Xp (B x Np, as ofdm_pilot_ls writes them) instead of grids.
#define MM_THREADS 128
__device__ __forceinline__ void block_sum4(double v[4], double (*red)[4]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = warp_sum(v[q]);
    __syncthreads();
    if (lane == 0) { red[w][0] = v[0]; red[w][1] = v[1]; red[w][2] = v[2]; red[w][3] = v[3]; }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) { double s = 0; for (int k = 0; k < MM_THREADS / 32; ++k) s += red[k][q]; v[q] = s; }
}

template <typename T, bool MEAS = false>
__global__ void __launch_bounds__(MM_THREADS) mmse_kernel(const cx<T>* __restrict__ grid, int64_t stream_stride, const int32_t* __restrict__ loc0,
                                                          const cx<T>* __restrict__ Xp, int Np, double Nps, int N_carrier, const cx<T>* __restrict__ h,
                                                          int h_len, const double* __restrict__ snr_db, PlanDev<T> p, cx<T>* __restrict__ H) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double red[MM_THREADS / 32][4];
    double2* t = (double2*)smem_raw;     // first column of Rpp: t[m] = 1/(1 + j*c*m), t[0] += 1/snr
    double2* Ht = t + Np;                // LS estimate at the pilots
    double2* f = Ht + Np;                // forward vector (two buffers)
    double2* f2 = f + Np;
    double2* x = f2 + Np;                // solution of Rpp x = Ht
    cx<T>* y = (cx<T>*)(x + Np);         // knots for the spline stage
    cx<T>* d = y + p.n_knots;
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x;
    const cx<T>* Y = grid + b * stream_stride;
    // tau_rms from the power-delay moments of h (:19-24)
    double v[4] = {0, 0, 0, 0};
    for (int k = tid; k < h_len; k += MM_THREADS) {
        double2 hv = to_d(h[b * h_len + k]);
        double pw = hv.x * hv.x + hv.y * hv.y;
        v[0] += pw; v[1] += pw * k; v[2] += pw * (double)k * (double)k;
    }
    block_sum4(v, red);
    const double r = v[1] / v[0], r2 = v[2] / v[0];
    const double tau_rms = sqrt(fmax(r2 - r * r, 0.0));
    const double c = 2.0 * CUDART_PI * tau_rms / (double)N_carrier * Nps;   // j2pi_tau_df*Nps = 1j*c
    const double snr = pow(10.0, snr_db[b] * 0.1);
    for (int m = tid; m < Np; m += MM_THREADS) {
        double den = 1.0 + c * c * (double)m * (double)m;    // 1/(1+j c m) = (1 - j c m)/den
        t[m] = make_double2(1.0 / den + (m == 0 ? 1.0 / snr : 0.0), -c * (double)m / den);
        Ht[m] = MEAS ? to_d(Y[m]) : to_d(cdiv(Y[loc0[m]], Xp[m]));   // :17 computed in T like LS_CE, promoted
    }
    __syncthreads();
    // Levinson: T[i][j] = t[i-j] (i>=j), conj(t[j-i]) otherwise.  f solves T_m f = e_1; the backward
    // vector is conj(reverse(f)).
    if (tid == 0) { f[0] = make_double2(1.0 / t[0].x, 0.0); x[0] = cscale(Ht[0], 1.0 / t[0].x); }
    __syncthreads();
    double2* fc = f; double2* fn = f2;
    for (int m = 1; m < Np; ++m) {
        // eps_f = sum_i t[m-i] f[i], eps_x = sum_i t[m-i] x[i]   (last row of T_{m+1} against [f;0], [x;0])
        double a[4] = {0, 0, 0, 0};
        for (int i = tid; i < m; i += MM_THREADS) {
            double2 tv = t[m - i];
            double2 e1 = cmul(tv, fc[i]), e2 = cmul(tv, x[i]);
            a[0] += e1.x; a[1] += e1.y; a[2] += e2.x; a[3] += e2.y;
        }
        block_sum4(a, red);
        const double2 ef = make_double2(a[0], a[1]), ex = make_double2(a[2], a[3]);
        const double den = 1.0 - (ef.x * ef.x + ef.y * ef.y);   // 1 - eps_f*eps_b, eps_b = conj(eps_f)
        // f_new = ([f;0] - eps_f*[0;b]) / den, b[i] = conj(f[m-1-i]);  b_new = conj(reverse(f_new))
        for (int i = tid; i <= m; i += MM_THREADS) {
            double2 fi = (i < m) ? fc[i] : make_double2(0, 0);
            double2 bi = (i >= 1) ? cconj(fc[m - i]) : make_double2(0, 0);
            double2 nv = fi - cmul(ef, bi);
            fn[i] = cscale(nv, 1.0 / den);
        }
        __syncthreads();
        // x_new = [x;0] + (Ht[m] - eps_x) * b_new,  b_new[i] = conj(f_new[m-i])
        const double2 g = Ht[m] - ex;
        for (int i = tid; i <= m; i += MM_THREADS) {
            double2 xi = (i < m) ? x[i] : make_double2(0, 0);
            x[i] = xi + cmul(g, cconj(fn[m - i]));
        }
        double2* tmp = fc; fc = fn; fn = tmp;
        __syncthreads();
    }
    for (int k = tid; k < Np; k += MM_THREADS) {
        double2 hm = Ht[k] - cscale(x[k], 1.0 / snr);
        y[p.ext_lo + k] = from_d<T>(hm);
    }
    __syncthreads();
    plan_apply(p, y, d, H + b * p.nq);
}

// ---- equalize_signal (`Task 5/equalize_signal.m:3-7`)
template <typename T>
__global__ void equalize_kernel(const cx<T>* __restrict__ grid, int64_t B, int S, int Nfft, const cx<T>* __restrict__ H, int h_stride, int Nc,
                                cx<T>* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * S * (int64_t)Nfft) return;
    int k = (int)(i % Nfft);
    int64_t b = i / ((int64_t)S * Nfft);
    out[i] = (k < Nc) ? cdiv(grid[i], H[b * h_stride + k]) : mk<T>(0, 0);
}

// ------------------------------------------------------------------------------------ host
extern "C" int ofdm_interpolate(ofdm_ctx* ctx, const void* Hp, int64_t B, const int32_t* loc, int Np, int N, int method, void* H) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, Hp && H && loc && Np >= 2 && N >= 2 && B >= 0, "bad argument");
    REQUIRE(ctx, method == OFDM_INTERP_LINEAR || method == OFDM_INTERP_SPLINE, "unknown method");
    const int32_t* l0; int rc = pilots0(ctx, loc, Np, N, &l0); if (rc) return rc;
    if (B == 0) return OFDM_OK;
    const InterpPlan* pl = ctx_plan(ctx, loc, Np, N, nullptr, N, method);
    REQUIRE(ctx, pl != nullptr, "plan construction failed");
    DISPATCH_T(ctx, {
        size_t smem = 2 * sizeof(cx<T>) * pl->n_knots;
        auto k = interpolate_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<(unsigned)B, CE_THREADS, smem, ctx->stream>>>((const cx<T>*)Hp, plan_dev<T>(pl), (cx<T>*)H);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_ls_ce(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, const int32_t* loc, int Np, const double* pv, int Nc, void* H) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && H && loc && pv && Np >= 2 && Nc >= 2 && S > 0 && B >= 0, "bad argument");
    const int32_t* l0; int rc = pilots0(ctx, loc, Np, std::min(Nfft * S, Nc), &l0); if (rc) return rc;
    if (B == 0) return OFDM_OK;
    const InterpPlan* pl = ctx_plan(ctx, loc, Np, Nc, nullptr, Nc, OFDM_INTERP_SPLINE);
    const void* xp = ofdm_upload_pilots(ctx, pv, Np);   // Xp(k), k = 1..Np: first column (linear indexing)
    REQUIRE(ctx, pl && xp, "plan construction failed");
    DISPATCH_T(ctx, {
        size_t smem = 2 * sizeof(cx<T>) * pl->n_knots;
        auto k = ls_ce_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<(unsigned)B, CE_THREADS, smem, ctx->stream>>>((const cx<T>*)grid, (int64_t)S * Nfft, l0, (const cx<T>*)xp, plan_dev<T>(pl), (cx<T>*)H);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- Y = RX(pilotCarriers, 1) ./ pilotValues(:, 1): the measurement vector handed to MP/OMP
// (`Task 5/Main_model_Task_5.m:191`, `Task5_part2.m:190`)
template <typename T>
__global__ void pilot_ls_kernel(const cx<T>* __restrict__ grid, int64_t stream_stride, int64_t B, const int32_t* __restrict__ loc0, int Np,
                                const cx<T>* __restrict__ xp, cx<T>* __restrict__ y) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * Np) return;
    const int64_t b = i / Np;
    const int q = (int)(i - b * Np);
    y[i] = cdiv(grid[b * stream_stride + loc0[q]], xp[q]);
}
extern "C" int ofdm_pilot_ls(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, const int32_t* loc, int Np, const double* pv, void* y) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && y && loc && pv && Np >= 1 && S > 0 && B >= 0, "bad argument");
    const int32_t* l0; int rc = pilots0(ctx, loc, Np, Nfft, &l0); if (rc) return rc;
    if (B == 0) return OFDM_OK;
    const void* xp = ofdm_upload_pilots(ctx, pv, Np);
    REQUIRE(ctx, xp != nullptr, "pilot upload failed");
    DISPATCH_T(ctx, { pilot_ls_kernel<T><<<(unsigned)cdiv64(B * Np, 256), 256, 0, ctx->stream>>>((const cx<T>*)grid, (int64_t)S * Nfft, B, l0, Np, (const cx<T>*)xp, (cx<T>*)y); });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_estimate_channel(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, const int32_t* allc, int Nq, const int32_t* pc, int Np,
                                     const double* pv, void* H, void* Hp) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && H && allc && pc && pv && Np >= 2 && Nq >= 1 && S > 0 && B >= 0, "bad argument");
    const int32_t* l0; int rc = pilots0(ctx, pc, Np, Nfft, &l0); if (rc) return rc;
    if (B == 0) return OFDM_OK;
    const InterpPlan* pl = ctx_plan(ctx, pc, Np, 0, allc, Nq, OFDM_INTERP_SPLINE);
    const void* xp = ofdm_upload_pilots(ctx, pv, (size_t)Np * S);
    REQUIRE(ctx, pl && xp, "plan construction failed");
    DISPATCH_T(ctx, {
        size_t smem = 2 * sizeof(cx<T>) * pl->n_knots;
        auto k = estimate_channel_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<(unsigned)B, CE_THREADS, smem, ctx->stream>>>((const cx<T>*)grid, S, Nfft, l0, (const cx<T>*)xp, plan_dev<T>(pl), (cx<T>*)H, (cx<T>*)Hp);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_mmse_ce(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, const int32_t* loc, int Np, const double* pv, int Nc,
                            const void* h, int h_len, const double* snr_db, void* H) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && H && loc && pv && h && snr_db && Np >= 2 && Nc >= Np && h_len >= 1 && S > 0 && B >= 0, "bad argument");
    const int32_t* l0; int rc = pilots0(ctx, loc, Np, std::min(Nfft, Nc), &l0); if (rc) return rc;
    if (B == 0) return OFDM_OK;
    const InterpPlan* pl = ctx_plan(ctx, loc, Np, Nc, nullptr, Nc, OFDM_INTERP_SPLINE);
    const void* xp = ofdm_upload_pilots(ctx, pv, Np);
    REQUIRE(ctx, pl && xp, "plan construction failed");
    DISPATCH_T(ctx, {
        size_t smem = 5 * sizeof(double2) * Np + 2 * sizeof(cx<T>) * pl->n_knots;
        REQUIRE(ctx, smem <= 220 * 1024, "too many pilots for the in-SMEM Levinson solver");
        auto k = mmse_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<(unsigned)B, MM_THREADS, smem, ctx->stream>>>((const cx<T>*)grid, (int64_t)S * Nfft, l0, (const cx<T>*)xp, Np, (double)(loc[1] - loc[0]), Nc,
                                                           (const cx<T>*)h, h_len, snr_db, plan_dev<T>(pl), (cx<T>*)H);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// MMSE_CE from measurement vectors (not exported): y_dev B x Np = RX(pilot_loc,1)./Xp, h_dev B x h_len, snr_db_dev B doubles.
// The same kernel as ofdm_mmse_ce with the quotient already taken, so the result is bit-identical to ofdm_mmse_ce on the grid
// that ofdm_pilot_ls read y from.  Used by ofdm_sweep_mse, whose front end hands out y only.
int ofdm_mmse_ce_meas(ofdm_ctx* ctx, const void* y, int64_t B, const int32_t* loc, int Np, int Nc, const void* h, int h_len, const double* snr_db,
                      void* H) {
    REQUIRE(ctx, y && H && loc && h && snr_db && Np >= 2 && Nc >= Np && h_len >= 1 && B >= 0, "bad argument");
    const int32_t* l0; int rc = pilots0(ctx, loc, Np, Nc, &l0); if (rc) return rc;
    if (B == 0) return OFDM_OK;
    const InterpPlan* pl = ctx_plan(ctx, loc, Np, Nc, nullptr, Nc, OFDM_INTERP_SPLINE);
    REQUIRE(ctx, pl != nullptr, "plan construction failed");
    DISPATCH_T(ctx, {
        size_t smem = 5 * sizeof(double2) * Np + 2 * sizeof(cx<T>) * pl->n_knots;
        REQUIRE(ctx, smem <= 220 * 1024, "too many pilots for the in-SMEM Levinson solver");
        auto k = mmse_kernel<T, true>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<(unsigned)B, MM_THREADS, smem, ctx->stream>>>((const cx<T>*)y, (int64_t)Np, l0, nullptr, Np, (double)(loc[1] - loc[0]), Nc,
                                                           (const cx<T>*)h, h_len, snr_db, plan_dev<T>(pl), (cx<T>*)H);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_equalize(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, const void* H, int h_stride, int Nc, void* out) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && H && out && S > 0 && B >= 0 && Nc >= 0 && Nc <= Nfft && h_stride >= Nc, "bad argument");
    if (B == 0) return OFDM_OK;
    int64_t n = B * S * (int64_t)Nfft;
    DISPATCH_T(ctx, { equalize_kernel<T><<<(unsigned)cdiv64(n, 256), 256, 0, ctx->stream>>>((const cx<T>*)grid, B, S, Nfft, (const cx<T>*)H, h_stride, Nc, (cx<T>*)out); });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}
