// OMP_estimate on tensor cores for large batches with a dense dictionary (SURVEY M4, `Task 5/OMP_estimate.m:7,14`):
// per iteration the correlation A^H r of ALL frames is one tcgen05 GEMM (TF32 in, FP32 accumulate in TMEM) whose
// epilogue keeps the 4 best |a_l^H r|^2 per frame (tc_gemm.cuh); a SIMT step kernel then re-scores those
// candidates in FP32/double, so the tensor cores only *screen* and the selected index is the exact FP32 argmax
// (frames whose TF32 top-4 is not clearly separated fall back to the exact full search).  The rest of the
// iteration -- pinv via the Gram matrix and a double Cholesky, residual, the 1e-2 stopping rule -- is the same
// arithmetic as the SIMT pursuit kernel in sparse.cu.
#include "pursuit_common.cuh"
#include "tc_gemm.cuh"

#define TS_THREADS 128
#define TS_DONE 0x40000000

// B operand: row 2l = [Re a_l | Im a_l], row 2l+1 = [-Im a_l | Re a_l], zero padded to K2 columns / 2*Lpad rows
__global__ void tc_dict_kernel(const float2* __restrict__ A, int Np, int Ldict, int K2, float* __restrict__ Bt) {
    const int l = blockIdx.x;
    float* r0 = Bt + (size_t)(2 * l) * K2;
    float* r1 = r0 + K2;
    for (int i = threadIdx.x; i < K2; i += blockDim.x) {
        float v0 = 0.f, v1 = 0.f;
        if (l < Ldict) {
            if (i < Np) { float2 a = A[(size_t)l * Np + i]; v0 = a.x; v1 = -a.y; }
            else if (i < 2 * Np) { float2 a = A[(size_t)l * Np + i - Np]; v0 = a.y; v1 = a.x; }
        }
        r0[i] = v0; r1[i] = v1;
    }
}
// A operand: row f = [Re r_f | Im r_f]; starts as the measurement
__global__ void tc_init_kernel(const float2* __restrict__ Y, int64_t B, int Np, int K2, float* __restrict__ Rt, int32_t* __restrict__ nsel) {
    const int64_t f = blockIdx.x;
    float* row = Rt + f * K2;
    for (int i = threadIdx.x; i < K2; i += blockDim.x) {
        float v = 0.f;
        if (f < B) { if (i < Np) v = Y[f * Np + i].x; else if (i < 2 * Np) v = Y[f * Np + i - Np].y; }
        row[i] = v;
    }
    if (threadIdx.x == 0 && f < B) nsel[f] = 0;
}

// sum N doubles per thread over the block (TS_THREADS = 4 warps): one pass of shuffles, two barriers
template <int N> __device__ __forceinline__ void block_sum_vec(double (&v)[N], double* sh /* 4*N */) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = warp_sum(v[k]);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < N; ++k) sh[w * N + k] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = (sh[k] + sh[N + k]) + (sh[2 * N + k] + sh[3 * N + k]);
    __syncthreads();
}

#define TS_MAXK 16
static_assert(TC_TOP == TS_THREADS / 32, "one warp re-scores one screened candidate");

// Hermitian positive (semi-)definite k x k solve G x = g in double by ONE WARP (all 32 lanes call; k <= TS_MAXK):
// lane i owns row i.  Column j of the factor needs the j previous columns, so the factorisation is k steps of O(j)
// work per lane instead of thread 0 walking k^3/3 terms alone; both triangular solves are right-looking (the lane
// that just finished an unknown broadcasts it, the others update their partial sums).  Same operations as
// chol_solve (pursuit_common.cuh); the backward solve accumulates in the opposite order.
static __device__ __forceinline__ void chol_solve_warp(int k, const double2 (*G)[TS_MAXK], const double2* g, double2* x, double2 (*Lm)[TS_MAXK]) {
    const int lane = threadIdx.x & 31;
    for (int j = 0; j < k; ++j) {
        if (lane == j) {
            double s = G[j][j].x;
            for (int q = 0; q < j; ++q) s -= Lm[j][q].x * Lm[j][q].x + Lm[j][q].y * Lm[j][q].y;
            Lm[j][j] = make_double2(sqrt(fmax(s, 0.0)), 0.0);
        }
        __syncwarp();
        const double dj = Lm[j][j].x;
        if (lane > j && lane < k) {
            double2 a = G[lane][j];
            for (int q = 0; q < j; ++q) a = a - cmulc(Lm[lane][q], Lm[j][q]);
            Lm[lane][j] = dj > 0 ? cscale(a, 1.0 / dj) : make_double2(0, 0);
        }
        __syncwarp();
    }
    double2 a = lane < k ? g[lane] : make_double2(0, 0);
    for (int i = 0; i < k; ++i) {                  // L z = g
        const double d = Lm[i][i].x;
        const double2 mine = d > 0 ? cscale(a, 1.0 / d) : make_double2(0, 0);
        const double2 zi = make_double2(__shfl_sync(0xffffffffu, mine.x, i), __shfl_sync(0xffffffffu, mine.y, i));
        if (lane == i) a = zi;
        else if (lane > i && lane < k) a = a - cmul(Lm[lane][i], zi);
    }
    for (int i = k - 1; i >= 0; --i) {             // L^H x = z
        const double d = Lm[i][i].x;
        const double2 mine = d > 0 ? cscale(a, 1.0 / d) : make_double2(0, 0);
        const double2 xi = make_double2(__shfl_sync(0xffffffffu, mine.x, i), __shfl_sync(0xffffffffu, mine.y, i));
        if (lane == i) a = xi;
        else if (lane < i) a = a - cmul(cconj(Lm[i][lane]), xi);
    }
    if (lane < k) x[lane] = a;
    __syncwarp();
}
// One OMP iteration for one frame.  Per-frame state lives in global memory between iterations: the selection list,
// the coefficients, the Gram matrix of the unique selected columns and its right-hand side (both double), and the
// residual (inside the GEMM's A operand).  The Gram matrix grows by one row per iteration.
__global__ void __launch_bounds__(TS_THREADS) omp_tc_step_kernel(const float2* __restrict__ Y, const float2* __restrict__ A, int Np, int Ldict, int K2, int it,
                                                                 const int32_t* __restrict__ cand, const float* __restrict__ cand_score,
                                                                 float* __restrict__ Rt, int32_t* __restrict__ sel_g, int32_t* __restrict__ nsel_g,
                                                                 float2* __restrict__ xs_g, double2* __restrict__ G_g, double2* __restrict__ rhs_g, int K,
                                                                 int32_t* __restrict__ fallbacks, int32_t* __restrict__ near_out, float tie_eps) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double shred[4 * 2 * (TS_MAXK + 2)];
    __shared__ float sval[32];
    __shared__ int sidx[32];
    __shared__ int sel[TS_MAXK], uniq[TS_MAXK], ucol[TS_MAXK], umult[TS_MAXK];
    __shared__ double2 G[TS_MAXK][TS_MAXK], Lm[TS_MAXK][TS_MAXK], grhs[TS_MAXK], xu[TS_MAXK];
    __shared__ float sc_m[TC_TOP];
    __shared__ int sc_c[TC_TOP];
    __shared__ int s_col, s_nu, s_new;
    const int64_t f = blockIdx.x;
    const int tid = threadIdx.x;
    int nsel = nsel_g[f];
    if (nsel & TS_DONE) return;                         // stopped by the 1e-2 rule in an earlier iteration
    float2* r = (float2*)smem_raw;
    float2* yv = r + Np;
    float* row = Rt + f * K2;
    for (int i = tid; i < Np; i += TS_THREADS) { r[i] = make_float2(row[i], row[Np + i]); yv[i] = Y[f * Np + i]; }
    if (tid < nsel) sel[tid] = sel_g[f * K + tid];
    __syncthreads();
    // ---- exact re-scoring of the screened candidates in one pass (first maximum wins, as MATLAB's max)
    {
        const float s0 = cand_score[f * TC_TOP], s3 = cand_score[f * TC_TOP + TC_TOP - 1];
        if (s3 < 0.995f * s0 && s0 > 0.f) {   // TF32 scores are good to ~2e-3: the exact argmax is then inside the top-4
            const int w = tid >> 5, lane = tid & 31;          // warp w scores candidate w
            const int clw = cand[f * TC_TOP + w];
            const float2* aw = A + (size_t)clw * Np;
            double ar = 0, ai = 0;
            for (int i = lane; i < Np; i += 32) { const double2 t = cmulc(to_d(r[i]), to_d(aw[i])); ar += t.x; ai += t.y; }   // conj(a) * r
            ar = warp_sum(ar); ai = warp_sum(ai);
            if (lane == 0) { sc_m[w] = (float)(ar * ar + ai * ai); sc_c[w] = clw; }
            __syncthreads();
            if (tid == 0) {
                float best = -CUDART_INF_F, sec = -CUDART_INF_F; int bi = 0x7fffffff;
#pragma unroll
                for (int c = 0; c < TC_TOP; ++c) {
                    const float m = sc_m[c];
                    if (m > best || (m == best && sc_c[c] < bi)) { sec = best; best = m; bi = sc_c[c]; } else if (m > sec) sec = m;
                }
                s_col = (bi == 0x7fffffff) ? 0 : bi;
                if (near_out && !(best - sec > tie_eps * best)) near_out[f] += 1;     // top-2 margin of the exact scores below tie_eps
            }
        } else {                                        // TF32 ranking too close to call: exact search over every column
            if (tid == 0 && fallbacks) atomicAdd(fallbacks, 1);
            float best = -CUDART_INF_F; int bi = 0x7fffffff;
            for (int l = tid; l < Ldict; l += TS_THREADS) {
                const float2* a = A + (size_t)l * Np;
                float ar = 0, ai = 0;
                for (int i = 0; i < Np; ++i) { float2 av = a[i], v = r[i]; ar += av.x * v.x + av.y * v.y; ai += av.x * v.y - av.y * v.x; }
                const float m = ar * ar + ai * ai;
                if (m > best) { best = m; bi = l; }
            }
            block_argmax(best, bi, sval, sidx);
            if (tid == 0) { s_col = (bi == 0x7fffffff) ? 0 : bi; if (near_out) near_out[f] += 1; }   // the screen itself could not separate them
        }
    }
    // ---- unique columns so far (duplicates share one unknown: pinv's minimum-norm split)
    if (tid == 0) {
        int nu = 0;
        for (int q = 0; q < nsel; ++q) {
            int slot = -1;
            for (int u = 0; u < nu; ++u) if (ucol[u] == sel[q]) slot = u;
            if (slot < 0) { ucol[nu] = sel[q]; umult[nu] = 1; uniq[q] = nu; ++nu; } else { umult[slot] += 1; uniq[q] = slot; }
        }
    }
    __syncthreads();
    if (tid == 0) {
        const int col = s_col;
        int nu = 0;
        for (int q = 0; q < nsel; ++q) nu = max(nu, uniq[q] + 1);
        int slot = -1;
        for (int u = 0; u < nu; ++u) if (ucol[u] == col) slot = u;
        sel[nsel] = col;
        if (slot < 0) { ucol[nu] = col; umult[nu] = 1; uniq[nsel] = nu; s_new = 1; ++nu; } else { umult[slot] += 1; uniq[nsel] = slot; s_new = 0; }
        s_nu = nu;
    }
    __syncthreads();
    const int nu = s_nu, col = s_col;
    nsel += 1;
    double2* Gf = G_g + f * (int64_t)K * K;
    double2* rf = rhs_g + f * (int64_t)K;
    // ---- the Gram matrix grows by one row (new unique column only): nu dots + the right-hand side, one reduction
    if (s_new) {                                        // nu dots with the unique columns (the last one is |a_new|^2) + conj(a_new) * y
        const int w = tid >> 5, lane = tid & 31;
        const float2* an = A + (size_t)col * Np;
        for (int j = w; j <= nu; j += TS_THREADS / 32) {
            const float2* aq = A + (size_t)ucol[j < nu ? j : 0] * Np;
            double ar = 0, ai = 0;
            for (int i = lane; i < Np; i += 32) {
                const double2 av = to_d(an[i]);
                const double2 t = j < nu ? cmulc(av, to_d(aq[i])) : cmulc(to_d(yv[i]), av);   // conj(a_q) * a_new | conj(a_new) * y
                ar += t.x; ai += t.y;
            }
            ar = warp_sum(ar); ai = warp_sum(ai);
            if (lane == 0) { if (j < nu) Gf[j * K + (nu - 1)] = make_double2(ar, ai); else rf[nu - 1] = make_double2(ar, ai); }
        }
        __syncthreads();
    }
    if (tid < nu * nu) { const int q = tid / nu, j = tid % nu; G[q][j] = (q <= j) ? Gf[q * K + j] : cconj(Gf[j * K + q]); }
    if (tid < nu) grhs[tid] = rf[tid];
    __syncthreads();
    if (tid < 32) {
        chol_solve_warp(nu, G, grhs, xu, Lm);           // x = pinv(A_sel) * y on the unique columns
        if (tid < nsel) { const double2 v = cscale(xu[uniq[tid]], 1.0 / (double)umult[uniq[tid]]); xs_g[f * K + tid] = make_float2((float)v.x, (float)v.y); }
        if (tid == 0) sel_g[f * K + nsel - 1] = col;
    }
    __syncthreads();
    // ---- residue = y - A*x and the stopping rule (`OMP_estimate.m:18-22`)
    double nrm[2] = {0, 0};
    for (int i = tid; i < Np; i += TS_THREADS) {
        double2 acc = to_d(yv[i]);
        for (int q = 0; q < nu; ++q) acc = acc - cmul(to_d(A[(size_t)ucol[q] * Np + i]), xu[q]);
        const double2 old = to_d(r[i]);
        nrm[0] += (acc.x - old.x) * (acc.x - old.x) + (acc.y - old.y) * (acc.y - old.y);
        nrm[1] += old.x * old.x + old.y * old.y;
        row[i] = (float)acc.x; row[Np + i] = (float)acc.y;
    }
    block_sum_vec<2>(nrm, shred);
    if (tid == 0) nsel_g[f] = nsel | ((it >= 1 && sqrt(nrm[0]) / sqrt(nrm[1]) < 1e-2) ? TS_DONE : 0);
}

// h(index(i1)) = x(i1) in selection order (later duplicates overwrite), H = fft(h) as a K-term sum
__global__ void __launch_bounds__(TS_THREADS) omp_tc_finish_kernel(const int32_t* __restrict__ sel_g, const int32_t* __restrict__ nsel_g, const float2* __restrict__ xs_g,
                                                                   int K, int Nfft, const float2* __restrict__ tw, float2* __restrict__ Hout,
                                                                   float2* __restrict__ hout, int32_t* __restrict__ index_out, int32_t* __restrict__ iters_out) {
    __shared__ int ucol[PU_MAXK];
    __shared__ float2 hval[PU_MAXK];
    __shared__ int s_nu;
    const int64_t f = blockIdx.x;
    const int tid = threadIdx.x;
    const int nsel = nsel_g[f] & ~TS_DONE;
    if (tid == 0) {
        int nu = 0;
        for (int q = 0; q < nsel; ++q) {
            const int c = sel_g[f * K + q];
            int slot = -1;
            for (int u = 0; u < nu; ++u) if (ucol[u] == c) slot = u;
            if (slot < 0) { slot = nu; ucol[nu++] = c; }
            hval[slot] = xs_g[f * K + q];
        }
        s_nu = nu;
        if (index_out) for (int q = 0; q < K; ++q) index_out[f * K + q] = q < nsel ? sel_g[f * K + q] + 1 : 0;
        if (iters_out) iters_out[f] = nsel;
    }
    __syncthreads();
    const int nu = s_nu, Nmask = Nfft - 1;
    if (hout) {
        float2* hb = hout + f * (int64_t)Nfft;
        for (int i = tid; i < Nfft; i += TS_THREADS) {
            float2 v = make_float2(0.f, 0.f);
            for (int u = 0; u < nu; ++u) if (ucol[u] == i) v = hval[u];
            hb[i] = v;
        }
    }
    if (Hout) {
        // H(m) = sum_u h_u W^{c_u m}.  With m = 64 a + b the twiddle is W^{64 c a} * W^{c b}: two 64-entry rows per
        // selected tap, read once from the table into shared memory (exact entries), instead of nu scattered table
        // reads per output bin.  (Nfft % 64 == 0 is required; other sizes take the direct form.)
        __shared__ float2 t_hi[TS_MAXK][64], t_lo[TS_MAXK][64];
        if ((Nfft & 63) == 0) {
            for (int e = tid; e < nu * 64; e += TS_THREADS) {
                const int u = e >> 6, j = e & 63;
                const float2 v = hval[u];
                const float2 w = tw[(64 * j * ucol[u]) & Nmask];
                t_hi[u][j] = make_float2(v.x * w.x - v.y * w.y, v.x * w.y + v.y * w.x);       // h_u * W^{64 c a}
                t_lo[u][j] = tw[(j * ucol[u]) & Nmask];
            }
            __syncthreads();
            for (int m = tid; m < Nfft; m += TS_THREADS) {
                const int a = m >> 6, bq = m & 63;
                float ar = 0, ai = 0;
                for (int u = 0; u < nu; ++u) { const float2 x = t_hi[u][a], w = t_lo[u][bq]; ar += x.x * w.x - x.y * w.y; ai += x.x * w.y + x.y * w.x; }
                Hout[f * (int64_t)Nfft + m] = make_float2(ar, ai);
            }
        } else {
            for (int m = tid; m < Nfft; m += TS_THREADS) {
                float ar = 0, ai = 0;
                for (int u = 0; u < nu; ++u) { float2 w = tw[(m * ucol[u]) & Nmask]; float2 v = hval[u]; ar += v.x * w.x - v.y * w.y; ai += v.x * w.y + v.y * w.x; }
                Hout[f * (int64_t)Nfft + m] = make_float2(ar, ai);
            }
        }
    }
}

// returns OFDM_OK and sets *handled when the tensor-core path ran
int ofdm_omp_tc(ofdm_ctx* ctx, const void* y, int64_t B, int Np, const void* A, int Ldict, int Nfft, int K, void* H, void* h, int32_t* index, int32_t* iters,
                int32_t* near_ties, double tie_eps, bool* handled) {
    *handled = false;
    if (ctx->precision != OFDM_PREC_F32 || !A || K > TS_MAXK) return OFDM_OK;
    if (getenv("OFDM_B200_NO_TC")) return OFDM_OK;
    const char* force = getenv("OFDM_B200_FORCE_TC");
    // a real dense contraction only: enough frames to fill 128-row tiles on every SM and a large dictionary
    if (!force && (B < 1024 || (int64_t)Np * Ldict < (1 << 18))) return OFDM_OK;
    if ((((uintptr_t)A) & 7) || (((uintptr_t)y) & 7)) return OFDM_OK;
    if (!tc_get_encode()) return OFDM_OK;
    const int K2 = ((2 * Np + TC_BK - 1) / TC_BK) * TC_BK;
    const int Lpad = ((Ldict + 63) / 64) * 64;
    const int64_t Bpad = ((B + TC_BM - 1) / TC_BM) * TC_BM;
    const void* tw = ctx_twiddles(ctx, Nfft);
    REQUIRE(ctx, tw != nullptr, "twiddle allocation failed");
    cudaStream_t st = ctx->stream;
    float *Bt = nullptr, *Rt = nullptr, *score = nullptr;
    int32_t *cand = nullptr, *sel = nullptr, *nsel = nullptr, *fb = nullptr;
    float2* xs = nullptr;
    double2 *Gs = nullptr, *rhs = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync((void**)&Bt, sizeof(float) * (size_t)2 * Lpad * K2, st));
    CUDA_TRY(ctx, cudaMallocAsync((void**)&Rt, sizeof(float) * (size_t)Bpad * K2, st));
    CUDA_TRY(ctx, cudaMallocAsync((void**)&score, sizeof(float) * (size_t)Bpad * TC_TOP, st));
    CUDA_TRY(ctx, cudaMallocAsync((void**)&cand, sizeof(int32_t) * (size_t)Bpad * TC_TOP, st));
    CUDA_TRY(ctx, cudaMallocAsync((void**)&sel, sizeof(int32_t) * (size_t)B * K, st));
    CUDA_TRY(ctx, cudaMallocAsync((void**)&nsel, sizeof(int32_t) * (size_t)(B + 1), st));
    CUDA_TRY(ctx, cudaMallocAsync((void**)&xs, sizeof(float2) * (size_t)B * K, st));
    CUDA_TRY(ctx, cudaMallocAsync((void**)&Gs, sizeof(double2) * (size_t)B * K * K, st));
    CUDA_TRY(ctx, cudaMallocAsync((void**)&rhs, sizeof(double2) * (size_t)B * K, st));
    fb = nsel + B;
    CUDA_TRY(ctx, cudaMemsetAsync(fb, 0, sizeof(int32_t), st));
    if (near_ties) CUDA_TRY(ctx, cudaMemsetAsync(near_ties, 0, sizeof(int32_t) * (size_t)B, st));
    tc_dict_kernel<<<Lpad, 128, 0, st>>>((const float2*)A, Np, Ldict, K2, Bt);
    tc_init_kernel<<<(unsigned)Bpad, 128, 0, st>>>((const float2*)y, B, Np, K2, Rt, nsel);
    ctx->launches += 2;
    CUtensorMap mapA, mapB;
    int rc = OFDM_OK;
    if (!tc_make_kmajor_map(&mapA, Rt, (uint64_t)Bpad, (uint64_t)K2) || !tc_make_kmajor_map(&mapB, Bt, (uint64_t)2 * Lpad, (uint64_t)K2))
        rc = ctx_fail(ctx, OFDM_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    if (rc == OFDM_OK) {
        func_smem_optin((const void*)tc_corr_top_kernel, TC_SMEM_TOP_BYTES);
        const size_t smem_step = sizeof(float2) * 2 * (size_t)Np;
        func_smem_optin((const void*)omp_tc_step_kernel, (int)std::max<size_t>(smem_step, 64 * 1024));
        for (int it = 0; it < K; ++it) {
            tc_corr_top_kernel<<<(unsigned)(Bpad / TC_BM), TC_THREADS, TC_SMEM_TOP_BYTES, st>>>(mapA, mapB, 2 * Lpad / TC_BN, K2, Ldict, cand, score);
            omp_tc_step_kernel<<<(unsigned)B, TS_THREADS, smem_step, st>>>((const float2*)y, (const float2*)A, Np, Ldict, K2, it, cand, score, Rt, sel, nsel, xs, Gs, rhs, K, fb, near_ties, (float)tie_eps);
            ctx->launches += 2;
        }
        omp_tc_finish_kernel<<<(unsigned)B, TS_THREADS, 0, st>>>(sel, nsel, xs, K, Nfft, (const float2*)tw, (float2*)H, (float2*)h, index, iters);
        ctx->launches++;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "tensor-core OMP launch failed: %s", cudaGetErrorString(e));
    }
    cudaFreeAsync(Bt, st); cudaFreeAsync(Rt, st); cudaFreeAsync(score, st); cudaFreeAsync(cand, st);
    cudaFreeAsync(sel, st); cudaFreeAsync(nsel, st); cudaFreeAsync(xs, st); cudaFreeAsync(Gs, st); cudaFreeAsync(rhs, st);
    if (rc == OFDM_OK) *handled = true;
    return rc;
}
