// OMP_estimate / MP_estimate: greedy sparse CIR recovery, one thread block per frame.
// Dictionary: dense (Np x Ldict, any complex matrix) or the partial-DFT descriptor
// A(i,l) = exp(-2*pi*1j*(p_i-1)*(l-1)/Nfft) of `Task 5/Main_model_Task_5.m:182-190`, for which
// A^H r = Nfft * ifft(scatter(r -> pilot bins))(1:Ldict) (SURVEY KAT 6) runs on the block FFT.
#include "fft.cuh"
#include "pursuit_common.cuh"

// dictionary element A(i, l)
template <typename T, bool DENSE>
__device__ __forceinline__ cx<T> dict_at(const cx<T>* __restrict__ At, int Ldict, const int32_t* __restrict__ p0, const cx<T>* __restrict__ tw,
                                         int Nmask, int i, int l) {
    if (DENSE) return At[(size_t)i * Ldict + l];
    return tw[(p0[i] * l) & Nmask];   // exp(-2j*pi*p*l/N); p*l < 2^31 for N <= 8192
}

template <typename T, bool DENSE, bool IS_OMP>
__global__ void __launch_bounds__(PU_THREADS) pursuit_kernel(const cx<T>* __restrict__ Y, int Np, const cx<T>* __restrict__ At, int Ldict,
                                                             const int32_t* __restrict__ p0, int Nfft, int logN, const cx<T>* __restrict__ tw,
                                                             const T* __restrict__ norms2, int K, cx<T>* __restrict__ Hout, cx<T>* __restrict__ hout,
                                                             int32_t* __restrict__ index_out, int32_t* __restrict__ iters_out,
                                                             int32_t* __restrict__ near_out, T tie_eps) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using C = cx<T>;
    __shared__ double red[32];
    __shared__ T sval[32];
    __shared__ int sidx[32];
    __shared__ int sel[PU_MAXK];          // selected columns (0-based), in selection order
    __shared__ int uniq[PU_MAXK];         // slot in the unique list for each selection
    __shared__ int ucol[PU_MAXK], umult[PU_MAXK];
    __shared__ double2 G[PU_MAXK][PU_MAXK], Lm[PU_MAXK][PU_MAXK], grhs[PU_MAXK], xu[PU_MAXK];
    __shared__ C xs[PU_MAXK];             // coefficient per selection (x(i1))
    __shared__ int s_stop, s_near;
    C* r = (C*)smem_raw;                  // residual
    C* yv = r + Np;                       // measurement
    C* fa = yv + Np;                      // FFT buffers (DFT path only)
    C* fb = fa + Nfft;
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x;
    const int Nmask = Nfft - 1;
    const int search = IS_OMP ? Ldict : min(Np, Ldict);   // `MP_estimate.m:3,10`: only the first Np columns
    for (int i = tid; i < Np; i += PU_THREADS) { C v = Y[b * Np + i]; r[i] = v; yv[i] = v; }
    if (tid == 0) { s_stop = 0; s_near = 0; }
    __syncthreads();
    int nsel = 0, nu = 0;
    for (int it = 0; it < K; ++it) {
        // ---- correlation + argmax
        T best = (T)-CUDART_INF, second = (T)-CUDART_INF; int bi = 0x7fffffff;
        if (DENSE) {
            for (int l = tid; l < search; l += PU_THREADS) {
                T ar = 0, ai = 0;
                for (int i = 0; i < Np; ++i) { C a = At[(size_t)i * Ldict + l]; C v = r[i]; ar += a.x * v.x + a.y * v.y; ai += a.x * v.y - a.y * v.x; }  // conj(a)*r
                T m = ar * ar + ai * ai;
                if (!IS_OMP) {
                    m = m / norms2[l];
                    for (int q = 0; q < nsel; ++q) if (sel[q] == l) m = (T)-100;
                }
                if (m > best) { second = best; best = m; bi = l; } else if (m > second) second = m;
            }
        } else {
            for (int i = tid; i < Nfft; i += PU_THREADS) fa[i] = mk<T>(0, 0);
            __syncthreads();
            for (int i = tid; i < Np; i += PU_THREADS) fa[p0[i]] = r[i];
            __syncthreads();
            C* c = block_fft<T, true>(fa, fb, Nfft, logN, tw);   // unnormalised inverse = A^H r
            for (int l = tid; l < search; l += PU_THREADS) {
                T m = cabs2(c[l]);
                if (!IS_OMP) {
                    m = m / (T)Np;                                // ||a||^2 = Np for unit-modulus columns
                    for (int q = 0; q < nsel; ++q) if (sel[q] == l) m = (T)-100;
                }
                if (m > best) { second = best; best = m; bi = l; } else if (m > second) second = m;
            }
        }
        const T my_best = best; const int my_bi = bi;
        block_argmax(best, bi, sval, sidx);
        const int col = (bi == 0x7fffffff) ? 0 : bi;   // all-NaN correlation: MATLAB's max returns index 1
        if (near_out && IS_OMP) {                      // runner-up over the block: near-tie count (top-2 margin below tie_eps, relative)
            T sec = (my_bi == bi) ? second : my_best;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { T ov = __shfl_xor_sync(0xffffffffu, sec, o); sec = ov > sec ? ov : sec; }
            __syncthreads();
            if ((tid & 31) == 0) sval[tid >> 5] = sec;
            __syncthreads();
            if (tid == 0) {
                T s2 = sval[0];
                for (int w = 1; w < PU_THREADS / 32; ++w) s2 = sval[w] > s2 ? sval[w] : s2;
                if (!(best - s2 > tie_eps * best)) s_near += 1;
            }
            __syncthreads();
        }
        // ---- bookkeeping of the selection (duplicates share one unknown: pinv's minimum-norm split)
        int slot = -1;
        for (int q = 0; q < nu; ++q) if (ucol[q] == col) slot = q;
        __syncthreads();
        if (tid == 0) {
            sel[nsel] = col;
            if (slot < 0) { ucol[nu] = col; umult[nu] = 1; uniq[nsel] = nu; } else { umult[slot] += 1; uniq[nsel] = slot; }
        }
        const bool is_new = slot < 0;
        if (is_new) slot = nu;
        __syncthreads();
        if (IS_OMP) {
            if (is_new) {
                // Gram row and right-hand side for the new unique column
                for (int q = 0; q <= nu; ++q) {
                    double2 acc = make_double2(0, 0);
                    for (int i = tid; i < Np; i += PU_THREADS) {
                        double2 aq = to_d(dict_at<T, DENSE>(At, Ldict, p0, tw, Nmask, i, ucol[q]));
                        double2 an = to_d(dict_at<T, DENSE>(At, Ldict, p0, tw, Nmask, i, col));
                        double2 t = cmulc(an, aq);               // conj(a_q) * a_new = G[q][new]
                        acc = acc + t;
                    }
                    acc = block_csum(acc, red);
                    if (tid == 0) { G[q][nu] = acc; G[nu][q] = cconj(acc); }
                }
                double2 acc = make_double2(0, 0);
                for (int i = tid; i < Np; i += PU_THREADS) {
                    double2 an = to_d(dict_at<T, DENSE>(At, Ldict, p0, tw, Nmask, i, col));
                    acc = acc + cmulc(to_d(yv[i]), an);           // conj(a) * y
                }
                acc = block_csum(acc, red);
                if (tid == 0) grhs[nu] = acc;
                nu += 1;
            }
            nsel += 1;
            __syncthreads();
            if (tid == 0) {
                chol_solve(nu, G, grhs, xu, Lm);                      // x = pinv(A)*y on the unique columns
                for (int q = 0; q < nsel; ++q) { double2 v = cscale(xu[uniq[q]], 1.0 / (double)umult[uniq[q]]); xs[q] = from_d<T>(v); }
            }
            __syncthreads();
            // residue = y - A*x ; stopping rule on ||r_i - r_{i-1}|| / ||r_{i-1}|| (`OMP_estimate.m:18-22`)
            double dn = 0, on = 0;
            for (int i = tid; i < Np; i += PU_THREADS) {
                double2 acc = to_d(yv[i]);
                for (int q = 0; q < nu; ++q) acc = acc - cmul(to_d(dict_at<T, DENSE>(At, Ldict, p0, tw, Nmask, i, ucol[q])), xu[q]);
                double2 old = to_d(r[i]);
                dn += (acc.x - old.x) * (acc.x - old.x) + (acc.y - old.y) * (acc.y - old.y);
                on += old.x * old.x + old.y * old.y;
                r[i] = from_d<T>(acc);
            }
            dn = block_sum(dn, red);
            on = block_sum(on, red);
            if (it >= 1 && sqrt(dn) / sqrt(on) < 1e-2) { if (tid == 0) s_stop = 1; }
            __syncthreads();
            if (s_stop) break;
        } else {
            // x(i1) = a'*residue/||a||^2 ; residue -= a*x(i1)  (`MP_estimate.m:21-23`)
            double2 acc = make_double2(0, 0);
            for (int i = tid; i < Np; i += PU_THREADS) acc = acc + cmulc(to_d(r[i]), to_d(dict_at<T, DENSE>(At, Ldict, p0, tw, Nmask, i, col)));
            acc = block_csum(acc, red);
            double n2 = DENSE ? (double)norms2[col] : (double)Np;
            double2 xv = cscale(acc, 1.0 / n2);
            if (tid == 0) xs[nsel] = from_d<T>(xv);
            for (int i = tid; i < Np; i += PU_THREADS) {
                double2 a = to_d(dict_at<T, DENSE>(At, Ldict, p0, tw, Nmask, i, col));
                r[i] = from_d<T>(to_d(r[i]) - cmul(a, xv));
            }
            if (is_new) nu += 1;
            nsel += 1;
            __syncthreads();
        }
    }
    __syncthreads();
    // ---- outputs: h(index(i1)) = x(i1) in selection order (later duplicates overwrite), H = fft(h)
    C* hb = hout ? hout + b * (int64_t)Nfft : nullptr;
    if (hb) for (int i = tid; i < Nfft; i += PU_THREADS) hb[i] = mk<T>(0, 0);
    __syncthreads();
    // effective value per unique column = the last selection that wrote it
    __shared__ C hval[PU_MAXK];
    if (tid == 0) {
        for (int q = 0; q < nsel; ++q) hval[uniq[q]] = xs[q];
        if (hb) for (int q = 0; q < nu; ++q) hb[ucol[q]] = hval[q];
        if (index_out) for (int q = 0; q < K; ++q) index_out[b * K + q] = q < nsel ? sel[q] + 1 : 0;
        if (iters_out) iters_out[b] = nsel;
        if (near_out) near_out[b] = s_near;
    }
    __syncthreads();
    if (Hout) {
        for (int m = tid; m < Nfft; m += PU_THREADS) {
            T ar = 0, ai = 0;
            for (int q = 0; q < nu; ++q) { C w = tw[(m * ucol[q]) & Nmask]; C v = hval[q]; ar += v.x * w.x - v.y * w.y; ai += v.x * w.y + v.y * w.x; }
            Hout[b * (int64_t)Nfft + m] = mk<T>(ar, ai);
        }
    }
}

// column-major (Np x Ldict) -> row-major [Np][Ldict], plus squared column norms
template <typename T>
__global__ void dict_prepare_kernel(const cx<T>* __restrict__ A, int Np, int Ldict, cx<T>* __restrict__ At, T* __restrict__ norms2) {
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= Ldict) return;
    double s = 0;
    for (int i = 0; i < Np; ++i) { cx<T> v = A[(size_t)l * Np + i]; At[(size_t)i * Ldict + l] = v; s += (double)v.x * v.x + (double)v.y * v.y; }
    norms2[l] = (T)s;
}

int ofdm_omp_tc(ofdm_ctx* ctx, const void* y, int64_t B, int Np, const void* A, int Ldict, int Nfft, int K, void* H, void* h, int32_t* index, int32_t* iters,
                int32_t* near_ties, double tie_eps, bool* handled);

template <bool IS_OMP>
static int pursuit_common(ofdm_ctx* ctx, const void* y, int64_t B, int Np, const void* A, int Ldict, const int32_t* loc, int Nfft, int K, void* H,
                          void* h, int32_t* index, int32_t* iters, int32_t* near_ties = nullptr, double tie_eps = 0.0) {
    REQUIRE(ctx, y && B >= 0 && Np >= 1 && Ldict >= 1 && K >= 1 && K <= PU_MAXK, "bad argument (K must be 1..32)");
    REQUIRE(ctx, is_pow2(Nfft) && Nfft >= 8 && Nfft <= (ctx->precision == OFDM_PREC_F64 ? 4096 : 8192), "unsupported Nfft");
    REQUIRE(ctx, Ldict <= Nfft, "dictionary wider than Nfft (indices address an Nfft-long CIR)");
    REQUIRE(ctx, A || loc, "need a dense dictionary or pilot locations");
    if (!IS_OMP) REQUIRE(ctx, Ldict >= Np, "MP_estimate indexes the first Np columns (needs Ldict >= Np)");
    if (B == 0) return OFDM_OK;
    const void* tw = ctx_twiddles(ctx, Nfft);
    REQUIRE(ctx, tw != nullptr, "twiddle allocation failed");
    const int32_t* p0 = nullptr;
    if (!A) {
        std::vector<int32_t> v(Np);
        for (int i = 0; i < Np; ++i) { REQUIRE(ctx, loc[i] >= 1 && loc[i] <= Nfft, "pilot index out of range"); v[i] = loc[i] - 1; }
        p0 = (const int32_t*)ctx_blob(ctx, v.data(), sizeof(int32_t) * Np);
        REQUIRE(ctx, p0 != nullptr, "device upload failed");
    }
    DISPATCH_T(ctx, {
        using C = cx<T>;
        C* At = nullptr; T* norms = nullptr;
        if (A) {
            CUDA_TRY(ctx, cudaMallocAsync((void**)&At, sizeof(C) * (size_t)Np * Ldict, ctx->stream));
            CUDA_TRY(ctx, cudaMallocAsync((void**)&norms, sizeof(T) * Ldict, ctx->stream));
            dict_prepare_kernel<T><<<(Ldict + 127) / 128, 128, 0, ctx->stream>>>((const C*)A, Np, Ldict, At, norms);
            ctx->launches++;
        }
        size_t smem = sizeof(C) * (2 * (size_t)Np + (A ? 0 : 2 * (size_t)Nfft));
        auto kd = pursuit_kernel<T, true, IS_OMP>;
        auto kf = pursuit_kernel<T, false, IS_OMP>;
        // static shared (Gram + Cholesky factor, ~34 KB) plus dynamic can pass 48 KB: always opt in
        CUDA_TRY(ctx, func_smem_optin((const void*)kd, (int)std::max<size_t>(smem, 64 * 1024)));
        CUDA_TRY(ctx, func_smem_optin((const void*)kf, (int)std::max<size_t>(smem, 64 * 1024)));
        if (A) kd<<<(unsigned)B, PU_THREADS, smem, ctx->stream>>>((const C*)y, Np, At, Ldict, nullptr, Nfft, ilog2(Nfft), (const C*)tw, norms, K, (C*)H, (C*)h, index, iters, near_ties, (T)tie_eps);
        else kf<<<(unsigned)B, PU_THREADS, smem, ctx->stream>>>((const C*)y, Np, nullptr, Ldict, p0, Nfft, ilog2(Nfft), (const C*)tw, nullptr, K, (C*)H, (C*)h, index, iters, near_ties, (T)tie_eps);
        ctx->launches++;
        if (A) { cudaFreeAsync(At, ctx->stream); cudaFreeAsync(norms, ctx->stream); }
    });
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return ctx_fail(ctx, OFDM_ERR_CUDA, "pursuit kernel launch failed: %s", cudaGetErrorString(e));
    return OFDM_OK;
}

int ofdm_omp_dft(ofdm_ctx* ctx, const void* y, int64_t B, int Np, const int32_t* p0_dev, int Ldict, int Nfft, int K, void* H, void* h, int32_t* index,
                 int32_t* iters, int32_t* near_ties, double tie_eps, bool* handled);
int ofdm_omp_probe_dft(ofdm_ctx* ctx, const void* A, int Np, int Ldict, int Nfft, int32_t** p0_out, bool* is_dft);

extern "C" int ofdm_omp(ofdm_ctx* ctx, const void* y, int64_t B, int Np, const void* A, int Ldict, const int32_t* loc, int Nfft, int K, void* H,
                        void* h, int32_t* index, int32_t* iters) {
    return ofdm_omp_ex(ctx, y, B, Np, A, Ldict, loc, Nfft, K, H, h, index, iters, nullptr, 0.0);
}

extern "C" int ofdm_omp_ex(ofdm_ctx* ctx, const void* y, int64_t B, int Np, const void* A, int Ldict, const int32_t* loc, int Nfft, int K, void* H,
                           void* h, int32_t* index, int32_t* iters, int32_t* near_ties, double tie_eps) {
    if (!ctx) return OFDM_ERR_INVALID;
    const bool sane = y && B > 0 && Np >= 1 && Ldict >= 1 && K >= 1 && K <= PU_MAXK && is_pow2(Nfft) && Nfft >= 8 && Nfft <= 8192 && Ldict <= Nfft;
    if (sane && ctx->precision == OFDM_PREC_F32) {
        // (1) partial-DFT dictionaries -- given as the descriptor, or recognised in a dense matrix -- take the Batch-OMP kernel
        //     (sparse_dft.cu): one FFT per frame instead of K dense correlations
        bool handled = false;
        if (!A && loc) {
            std::vector<int32_t> v(Np);
            for (int i = 0; i < Np; ++i) { REQUIRE(ctx, loc[i] >= 1 && loc[i] <= Nfft, "pilot index out of range"); v[i] = loc[i] - 1; }
            const int32_t* p0 = (const int32_t*)ctx_blob(ctx, v.data(), sizeof(int32_t) * Np);
            REQUIRE(ctx, p0 != nullptr, "device upload failed");
            int rc = ofdm_omp_dft(ctx, y, B, Np, p0, Ldict, Nfft, K, H, h, index, iters, near_ties, tie_eps, &handled);
            if (rc || handled) return rc;
        } else if (A && B >= 64 && !getenv("OFDM_B200_NO_DFT_PROBE")) {
            int32_t* p0 = nullptr;
            bool is_dft = false;
            int rc = ofdm_omp_probe_dft(ctx, A, Np, Ldict, Nfft, &p0, &is_dft);
            if (rc) return rc;
            if (is_dft) {
                rc = ofdm_omp_dft(ctx, y, B, Np, p0, Ldict, Nfft, K, H, h, index, iters, near_ties, tie_eps, &handled);
                cudaFreeAsync(p0, ctx->stream);
                if (rc || handled) return rc;
            }
        }
        // (2) unstructured dense dictionaries in large batches: correlation on tcgen05 tensor cores (sparse_tc.cu)
        if (A) {
            int rc = ofdm_omp_tc(ctx, y, B, Np, A, Ldict, Nfft, K, H, h, index, iters, near_ties, tie_eps, &handled);
            if (rc || handled) return rc;
        }
    }
    return pursuit_common<true>(ctx, y, B, Np, A, Ldict, loc, Nfft, K, H, h, index, iters, near_ties, tie_eps);
}
extern "C" int ofdm_mp(ofdm_ctx* ctx, const void* y, int64_t B, int Np, const void* A, int Ldict, const int32_t* loc, int Nfft, int K, void* H,
                       void* h, int32_t* index) {
    if (!ctx) return OFDM_ERR_INVALID;
    return pursuit_common<false>(ctx, y, B, Np, A, Ldict, loc, Nfft, K, H, h, index, nullptr);
}
