// add_STO / add_CFO / Noise / get_MP_channel_resp + conv -- impairments on B x L serial streams.
#include "fft.cuh"
#include "philox.cuh"

int ofdm_stream_power_sum(ofdm_ctx* ctx, const void* in, int64_t B, int64_t L, double* power_sum);

// ---- add_STO (`Task 5/add_STO.m:5-9`)
template <typename T>
__global__ void add_sto_kernel(const cx<T>* __restrict__ in, int64_t B, int64_t L, const int32_t* __restrict__ nsto, cx<T>* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * L) return;
    int64_t b = i / L, n = i - b * L;
    int64_t src = n + (int64_t)nsto[b];
    out[i] = (src >= 0 && src < L) ? in[b * L + src] : mk<T>(0, 0);
}
extern "C" int ofdm_add_sto(ofdm_ctx* ctx, const void* in, int64_t B, int64_t L, const int32_t* nsto, void* out) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, in && out && nsto && B >= 0 && L >= 0 && in != out, "bad argument (in-place not supported)");
    if (B * L == 0) return OFDM_OK;
    DISPATCH_T(ctx, { add_sto_kernel<T><<<(unsigned)cdiv64(B * L, 256), 256, 0, ctx->stream>>>((const cx<T>*)in, B, L, nsto, (cx<T>*)out); });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- add_CFO (`Task 5/add_CFO.m:6-7`): y .* exp(2j*pi*CFO*n/Nfft).
// The rotation of sample n is DEFINED here as the double-precision product R(256 (n >> 8)) * R(n & 255), R(k) =
// exp(2j*pi*frac(CFO*k/Nfft)) with the phase range-reduced in double, rounded to the stream type once: one sincospi per 256
// samples and per thread instead of one per sample, and the fused Task-4 channel below uses the same definition, so both
// give identical bits.  (Against the direct evaluation the factor differs by < 3e-16 before the rounding.)
__device__ __forceinline__ double2 cfo_rot_d(double cfo, double inv_nfft, int64_t k) {
    double ph = cfo * (double)k * inv_nfft;
    ph -= floor(ph);
    double sn, cs;
    sincospi(2.0 * ph, &sn, &cs);
    return make_double2(cs, sn);
}
// (explicit rounding intrinsics: the contraction into FMAs is pinned, not left to each kernel's optimiser)
__device__ __forceinline__ float2 cmul_pinned(float2 v, float2 w) {
    return make_float2(__fmaf_rn(v.x, w.x, -__fmul_rn(v.y, w.y)), __fmaf_rn(v.x, w.y, __fmul_rn(v.y, w.x)));
}
__device__ __forceinline__ double2 cmul_pinned(double2 v, double2 w) {
    return make_double2(__fma_rn(v.x, w.x, -__dmul_rn(v.y, w.y)), __fma_rn(v.x, w.y, __dmul_rn(v.y, w.x)));
}
template <typename T>
__device__ __forceinline__ cx<T> cfo_rot_apply(cx<T> v, double2 rq, double2 rt) {
    const double2 r = cmul_pinned(rq, rt);
    return cmul_pinned(v, mk<T>((T)r.x, (T)r.y));
}
#define CFO_TILE 2048
template <typename T>
__global__ void __launch_bounds__(256) add_cfo_kernel(const cx<T>* __restrict__ in, int64_t L, const double* __restrict__ cfo, double inv_nfft, cx<T>* __restrict__ out) {
    __shared__ double2 rq[CFO_TILE / 256];
    const int64_t b = blockIdx.x, n0 = (int64_t)blockIdx.y * CFO_TILE;
    const double c = cfo[b];
    if (threadIdx.x < CFO_TILE / 256) rq[threadIdx.x] = cfo_rot_d(c, inv_nfft, n0 + 256 * threadIdx.x);
    const double2 rt = cfo_rot_d(c, inv_nfft, threadIdx.x);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < CFO_TILE / 256; ++i) {
        const int64_t n = n0 + 256 * i + threadIdx.x;
        if (n < L) out[b * L + n] = cfo_rot_apply<T>(in[b * L + n], rq[i], rt);
    }
}
extern "C" int ofdm_add_cfo(ofdm_ctx* ctx, const void* in, int64_t B, int64_t L, const double* cfo, int Nfft, void* out) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, in && out && cfo && B >= 0 && L >= 0 && Nfft > 0, "bad argument");
    if (B * L == 0) return OFDM_OK;
    REQUIRE(ctx, cdiv64(L, CFO_TILE) <= 65535, "stream too long");
    DISPATCH_T(ctx, { add_cfo_kernel<T><<<dim3((unsigned)B, (unsigned)cdiv64(L, CFO_TILE)), 256, 0, ctx->stream>>>((const cx<T>*)in, L, cfo, 1.0 / Nfft, (cx<T>*)out); });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- Noise (`Task 5/Noise.m:3-11`): mean power over the whole stream (double), then
// sqrt(P/2)*(N1 + 1i*N2).  N1/N2 imported (real block, imaginary block) or Philox.
// Deterministic: block y of stream b writes its partial sum, a second kernel adds the partials in a fixed order (no floating-point
// atomics: two calls on the same stream give the same sigma to the last bit, in FP64 mode too).
#define POWER_MAX_BLOCKS 64
template <typename T>
__global__ void stream_power_kernel(const cx<T>* __restrict__ in, int64_t L, double* __restrict__ partial) {
    __shared__ double red[32];
    const int64_t b = blockIdx.x;
    double s = 0;
    for (int64_t n = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; n < L; n += (int64_t)gridDim.y * blockDim.x) {
        cx<T> v = in[b * L + n];
        s += (double)v.x * (double)v.x + (double)v.y * (double)v.y;
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) partial[b * gridDim.y + blockIdx.y] = s;
}
__global__ void stream_power_finish_kernel(const double* __restrict__ partial, int64_t B, int nb, double* __restrict__ power_sum) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double s = 0;
    for (int y = 0; y < nb; ++y) s += partial[b * nb + y];
    power_sum[b] = s;
}
template <typename T>
__global__ void add_noise_kernel(const cx<T>* __restrict__ in, int64_t B, int64_t L, const double* __restrict__ snr_db,
                                 const double* __restrict__ power_sum, const T* __restrict__ normals, uint64_t seed,
                                 int64_t first_stream, cx<T>* __restrict__ out, double* __restrict__ nvar) {
    __shared__ T sigma_s;
    const int64_t b = blockIdx.x;
    if (threadIdx.x == 0) {                          // NoisePower = P / 10^(SNR/10), once per CTA (`Noise.m:3-5`)
        const double P = power_sum[b] / (double)L;
        const double np = P / pow(10.0, snr_db[b] / 10.0);
        sigma_s = (T)sqrt(np / 2);
        if (nvar && blockIdx.y == 0) nvar[b] = sqrt(np);
    }
    __syncthreads();
    const T sigma = sigma_s;
    if (normals) {
        for (int64_t n = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; n < L; n += (int64_t)gridDim.y * blockDim.x) {
            const T g1 = normals[(b * 2) * L + n], g2 = normals[(b * 2 + 1) * L + n];
            const cx<T> v = in[b * L + n];
            out[b * L + n] = mk<T>(v.x + sigma * g1, v.y + sigma * g2);
        }
    } else {                                         // one Philox call serves two consecutive samples
        for (int64_t pr = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; 2 * pr < L; pr += (int64_t)gridDim.y * blockDim.x) {
            float g[4];
            philox_normal_quad(seed, (uint64_t)(first_stream + b), (uint64_t)pr, g);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int64_t n = 2 * pr + e;
                if (n < L) { const cx<T> v = in[b * L + n]; out[b * L + n] = mk<T>(v.x + sigma * (T)g[2 * e], v.y + sigma * (T)g[2 * e + 1]); }
            }
        }
    }
}
extern "C" int ofdm_add_noise(ofdm_ctx* ctx, const void* in, int64_t B, int64_t L, const double* snr_db, const void* normals,
                              uint64_t seed, int64_t first_stream_id, void* out, double* nvar) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, in && out && snr_db && B >= 0 && L >= 0, "bad argument");
    if (B * L == 0) return OFDM_OK;
    double* psum = (double*)ctx_scratch(ctx, sizeof(double) * B);
    REQUIRE(ctx, psum != nullptr, "scratch allocation failed");
    {
        int rc = ofdm_stream_power_sum(ctx, in, B, L, psum);
        if (rc) return rc;
    }
    DISPATCH_T(ctx, {
        add_noise_kernel<T><<<dim3((unsigned)B, (unsigned)std::min<int64_t>(cdiv64(L, 256 * 4), 256)), 256, 0, ctx->stream>>>(
            (const cx<T>*)in, B, L, snr_db, psum, (const T*)normals, seed, first_stream_id, (cx<T>*)out, nvar);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- get_MP_channel_resp (`Task 5/get_MP_channel_resp.m:2-19`)
template <typename T>
__global__ void load_real_taps_kernel(const double* __restrict__ h, int D, int N, cx<T>* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = mk<T>(i < D ? (T)h[i] : (T)0, (T)0);
}
extern "C" int ofdm_mp_channel_resp(ofdm_ctx* ctx, const double* taps, int K, int Nfft, double* h_host, int h_cap, int* h_len, void* H_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, taps && K > 0 && h_host && h_len, "bad argument");
    int max_delay = 0;
    for (int i = 0; i < K; ++i) { REQUIRE(ctx, taps[2 * i] >= 0, "negative delay"); max_delay = std::max(max_delay, (int)taps[2 * i]); }
    int D = max_delay + 1;
    REQUIRE(ctx, D <= h_cap, "h_host too small");
    for (int i = 0; i < D; ++i) h_host[i] = 0;
    for (int i = 0; i < K; ++i) h_host[(int)taps[2 * i]] = taps[2 * i + 1];  // later rows overwrite (:14)
    *h_len = D;
    if (H_dev) {
        REQUIRE(ctx, D <= Nfft, "impulse response longer than Nfft");  // fft(h, Nfft) would truncate
        const double* hd = (const double*)ctx_blob(ctx, h_host, sizeof(double) * D);
        REQUIRE(ctx, hd != nullptr, "device upload failed");
        size_t esz = ctx->precision == OFDM_PREC_F64 ? sizeof(double2) : sizeof(float2);
        void* tmp = ctx_scratch(ctx, esz * Nfft);
        REQUIRE(ctx, tmp != nullptr, "scratch allocation failed");
        DISPATCH_T(ctx, { load_real_taps_kernel<T><<<(Nfft + 255) / 256, 256, 0, ctx->stream>>>(hd, D, Nfft, (cx<T>*)tmp); });
        LAUNCH_CHECK(ctx);
        return ofdm_fft(ctx, tmp, H_dev, 1, Nfft, 0);
    }
    return OFDM_OK;
}

// ---- conv(x, h, 'full')(1:L) (`Task 5/Main_model_Task_5.m:126-127`): short FIR, taps in shared memory.
template <typename T>
__global__ void fir_kernel(const cx<T>* __restrict__ in, int64_t B, int64_t L, const cx<T>* __restrict__ h, int D, int per_stream,
                           cx<T>* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* hv = (cx<T>*)smem_raw;                   // non-zero taps in ascending delay (sparse channels: 3-6 of 11-26)
    int* hd = (int*)(hv + D);
    __shared__ int nnz_s;
    const int64_t b = blockIdx.x;
    const cx<T>* hb = per_stream ? h + b * D : h;
    if (threadIdx.x == 0) {
        int k = 0;
        for (int d = 0; d < D; ++d) { const cx<T> t = hb[d]; if (t.x != (T)0 || t.y != (T)0) { hv[k] = t; hd[k] = d; ++k; } }
        nnz_s = k;
    }
    __syncthreads();
    const int nnz = nnz_s;
    const cx<T>* x = in + b * L;
    for (int64_t n = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; n < L; n += (int64_t)gridDim.y * blockDim.x) {
        cx<T> acc = mk<T>(0, 0);
        for (int t = 0; t < nnz; ++t) {
            const int d = hd[t];
            if ((int64_t)d <= n) acc = cmac(acc, x[n - d], hv[t]);
        }
        out[b * L + n] = acc;
    }
}
extern "C" int ofdm_apply_fir(ofdm_ctx* ctx, const void* in, int64_t B, int64_t L, const void* h, int D, int per_stream, void* out) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, in && out && h && B >= 0 && L >= 0 && D > 0 && in != out, "bad argument (in-place not supported)");
    REQUIRE(ctx, D <= 4096, "FIR longer than 4096 taps");
    if (B * L == 0) return OFDM_OK;
    int bx = (int)std::min<int64_t>(cdiv64(L, 256), 256);
    DISPATCH_T(ctx, {
        fir_kernel<T><<<dim3((unsigned)B, bx), 256, (sizeof(cx<T>) + sizeof(int)) * D, ctx->stream>>>((const cx<T>*)in, B, L, (const cx<T>*)h, D, per_stream, (cx<T>*)out);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- fused Task-5 channel: AWGN then FIR (`Task 5/Main_model_Task_5.m:108,123-127`).
// One CTA produces CH_TILE consecutive output samples of one stream: the noisy samples it needs (tile + D-1 of
// history) are formed in shared memory -- x + sigma*(g1 + i g2), the Philox normals are addressed by sample index,
// so the history of a tile is regenerated, not exchanged -- and filtered from there with the NON-ZERO taps only
// (ordered list built per CTA; the course's channels have 3-6 taps over 11-26 delays).  Same operations in the
// same order as add_noise_kernel followed by fir_kernel, without the 8 B/sample round trip in between.
#define CH_TILE 2048
#define CH_MAXD 1024
#define CH_CHUNK 8         // tiles per CTA
// Once per call: sigma of every stream (`Noise.m:3-5`: NoisePower = P / 10^(SNR/10), sigma = sqrt(NoisePower/2)) and
// the ordered list of non-zero taps, so that the 250k tile CTAs of a sweep point start straight into the generator.
template <typename T>
__global__ void channel_prep_kernel(int64_t B, int64_t L, const double* __restrict__ snr_db, const double* __restrict__ power_sum,
                                    const cx<T>* __restrict__ h, int D, T* __restrict__ sigma, cx<T>* __restrict__ hv, int* __restrict__ hd,
                                    int* __restrict__ nnz) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) {
        const double P = power_sum[b] / (double)L;
        sigma[b] = (T)sqrt(P / pow(10.0, snr_db[b] / 10.0) / 2);
    }
    if (b == 0) {
        int k = 0;
        for (int d = 0; d < D; ++d) { const cx<T> t = h[d]; if (t.x != (T)0 || t.y != (T)0) { hv[k] = t; hd[k] = d; ++k; } }
        *nnz = k;
    }
}
// IMP = true is the Task-4 order (`Task 4/Main_model_Task_4.m:95,103,110,263-264`): Noise -> add_STO -> add_CFO -> multipath.
// The staged sample m is then  rot(m) * noisy(m + nsto)  (zero where the shifted index leaves the stream, `add_STO.m:5-9`), the
// Philox normals stay addressed by the ORIGINAL sample index and rot(m) is add_cfo_kernel's two-level rotation: the same
// bits as ofdm_add_noise -> ofdm_add_sto -> ofdm_add_cfo -> ofdm_apply_fir in one pass over the signal.
template <typename T, bool IMP>
__global__ void __launch_bounds__(256) channel_t5_kernel(const cx<T>* __restrict__ in, int64_t L, const T* __restrict__ sigma_g, const T* __restrict__ normals,
                                                         uint64_t seed, int64_t first_stream, const cx<T>* __restrict__ hv_g, const int* __restrict__ hd_g,
                                                         const int* __restrict__ nnz_g, int D, cx<T>* __restrict__ out,
                                                         const int32_t* __restrict__ nsto_g, const double* __restrict__ cfo_g, double inv_nfft) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* sn = (cx<T>*)smem_raw;                   // D - 1 noisy samples of history, then the CH_TILE of the current tile
    cx<T>* hv = sn + CH_TILE + D - 1;               // non-zero taps, ascending delay
    int* hd = (int*)(hv + D);
    __shared__ double2 rq_s[CH_TILE / 256 + 2];     // IMP: R(256 q) for the q values of the current tile (+ one either side)
    const int64_t b = blockIdx.x;
    const int64_t c0 = (int64_t)blockIdx.y * CH_CHUNK * CH_TILE;    // this CTA walks CH_CHUNK consecutive tiles, carrying the history
    const T sigma = sigma_g[b];
    const int64_t sto = IMP ? (int64_t)nsto_g[b] : 0;
    const double cfo = IMP ? cfo_g[b] : 0.0;
    const int nnz = *nnz_g;
    for (int t = threadIdx.x; t < nnz; t += 256) { hv[t] = hv_g[t]; hd[t] = hd_g[t]; }
    const cx<T>* xin = in + b * L;
    const T* nre = normals ? normals + (b * 2) * L : nullptr;
    const T* nim = normals ? normals + (b * 2 + 1) * L : nullptr;
    const uint64_t sid = (uint64_t)(first_stream + b);
    // noisy sample n (0 outside the stream): x + sigma*(g1 + i g2), imported normals or the pair's Philox quad
    auto noisy_imported = [&](int64_t n) -> cx<T> {
        if (n < 0 || n >= L) return mk<T>(0, 0);
        const cx<T> x = xin[n];
        return mk<T>(x.x + sigma * nre[n], x.y + sigma * nim[n]);
    };
    auto noisy_pair = [&](int64_t pr, cx<T>& v0, cx<T>& v1) {          // samples 2 pr and 2 pr + 1 from one Philox call
        v0 = mk<T>(0, 0); v1 = mk<T>(0, 0);
        if (pr < 0 || 2 * pr >= L) return;
        float g[4];
        philox_normal_quad(seed, sid, (uint64_t)pr, g);
        const cx<T> x0 = xin[2 * pr];
        v0 = mk<T>(x0.x + sigma * (T)g[0], x0.y + sigma * (T)g[1]);
        if (2 * pr + 1 < L) { const cx<T> x1 = xin[2 * pr + 1]; v1 = mk<T>(x1.x + sigma * (T)g[2], x1.y + sigma * (T)g[3]); }
    };
    // IMP: staged sample m, evaluated on its own (history of the first tile, and every sample when the normals are imported)
    auto staged_imp = [&](int64_t m) -> cx<T> {
        const int64_t q = m + sto;
        if (m < 0 || m >= L || q < 0 || q >= L) return mk<T>(0, 0);
        cx<T> v;
        if (normals) v = noisy_imported(q);
        else {
            float g[4];
            philox_normal_quad(seed, sid, (uint64_t)(q >> 1), g);
            const cx<T> x = xin[q];
            v = (q & 1) ? mk<T>(x.x + sigma * (T)g[2], x.y + sigma * (T)g[3]) : mk<T>(x.x + sigma * (T)g[0], x.y + sigma * (T)g[1]);
        }
        return cfo_rot_apply<T>(v, cfo_rot_d(cfo, inv_nfft, (m >> 8) << 8), cfo_rot_d(cfo, inv_nfft, m & 255));
    };
    // history of the first tile: samples c0 - (D-1) .. c0 - 1 (regenerated, not exchanged; c0 is even)
    if (IMP) {
        for (int j = threadIdx.x; j < D - 1; j += 256) sn[j] = staged_imp(c0 - (D - 1) + j);
    } else if (normals) {
        for (int j = threadIdx.x; j < D - 1; j += 256) sn[j] = noisy_imported(c0 - (D - 1) + j);
    } else {
        for (int q = threadIdx.x; 2 * q < D - 1; q += 256) {            // pair c0/2 - 1 - q covers samples c0 - 2q - 2, c0 - 2q - 1
            cx<T> v0, v1;
            noisy_pair((c0 >> 1) - 1 - q, v0, v1);
            const int j1 = D - 2 - 2 * q;                               // slot of sample c0 - 2q - 1
            sn[j1] = v1;
            if (j1 >= 1) sn[j1 - 1] = v0;
        }
    }
    cx<T>* cur = sn + (D - 1);
    for (int tile = 0; tile < CH_CHUNK; ++tile) {
        const int64_t n0 = c0 + (int64_t)tile * CH_TILE;
        if (n0 >= L) break;
        const bool whole = n0 + CH_TILE <= L;               // no range test inside a whole tile
        if (IMP && normals) {
#pragma unroll
            for (int i = 0; i < CH_TILE / 256; ++i) cur[threadIdx.x + 256 * i] = staged_imp(n0 + threadIdx.x + 256 * i);
        } else if (IMP) {
            // Philox pairs over the SOURCE index: pair P0 + j holds source samples qb - par + 2 j and the next one, i.e. tile
            // slots l = 2 j - par and l + 1 (par = parity of qb = n0 + sto); j = 0 .. CH_TILE / 2 covers every slot once.
            // Slot l of this thread is 2 tid - par + e + 512 i: its (m & 255) part does not depend on i, so the two R(t) are
            // evaluated once per tile and the R(256 q) come from a small shared table.
            const int64_t qb = n0 + sto;
            const int par = (int)(qb & 1);
            const int64_t P0 = (qb - par) >> 1;
            __syncthreads();                                 // (rq_s of the previous tile is no longer read)
            if (threadIdx.x < CH_TILE / 256 + 2) rq_s[threadIdx.x] = cfo_rot_d(cfo, inv_nfft, n0 + 256 * ((int64_t)threadIdx.x - 1));
            const int la = 2 * (int)threadIdx.x - par;       // slot of element 0 at i = 0 (-1 for thread 0 when par = 1)
            const double2 rt0 = cfo_rot_d(cfo, inv_nfft, (la) & 255), rt1 = cfo_rot_d(cfo, inv_nfft, (la + 1) & 255);
            __syncthreads();
            for (int i = 0; i <= CH_TILE / 512; ++i) {
                const int j = threadIdx.x + 256 * i;
                if (j > CH_TILE / 2) break;
                const int64_t pr = P0 + j;
                float g[4] = {0.f, 0.f, 0.f, 0.f};
                if (pr >= 0 && 2 * pr < L) philox_normal_quad(seed, sid, (uint64_t)pr, g);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int l = la + e + 512 * i;
                    if (l < 0 || l >= CH_TILE) continue;
                    const int64_t q = 2 * pr + e, m = n0 + l;
                    cx<T> v = mk<T>(0, 0);
                    if (q >= 0 && q < L && m < L) {
                        const cx<T> x = xin[q];
                        v = cfo_rot_apply<T>(mk<T>(x.x + sigma * (T)g[2 * e], x.y + sigma * (T)g[2 * e + 1]), rq_s[(l >> 8) + 1], e ? rt1 : rt0);
                    }
                    cur[l] = v;
                }
            }
        } else if (normals) {
#pragma unroll
            for (int i = 0; i < CH_TILE / 256; ++i) cur[threadIdx.x + 256 * i] = noisy_imported(n0 + threadIdx.x + 256 * i);
        } else if (whole) {
            const cx<T>* xp = xin + n0;
            const uint64_t pr0 = (uint64_t)(n0 >> 1);
#pragma unroll
            for (int i = 0; i < CH_TILE / 512; ++i) {
                const int q = threadIdx.x + 256 * i;
                float g[4];
                philox_normal_quad(seed, sid, pr0 + (uint64_t)q, g);
                const cx<T> x0 = xp[2 * q], x1 = xp[2 * q + 1];
                cur[2 * q] = mk<T>(x0.x + sigma * (T)g[0], x0.y + sigma * (T)g[1]);
                cur[2 * q + 1] = mk<T>(x1.x + sigma * (T)g[2], x1.y + sigma * (T)g[3]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < CH_TILE / 512; ++i) {
                const int q = threadIdx.x + 256 * i;
                cx<T> v0, v1;
                noisy_pair((n0 >> 1) + q, v0, v1);
                cur[2 * q] = v0; cur[2 * q + 1] = v1;
            }
        }
        __syncthreads();
        // eight outputs per thread; the tap loop is outermost so that a tap is fetched once for all of them (the order of
        // additions per output is still ascending delay).  Samples before the start of the stream are absent, not zero.
        cx<T> acc[CH_TILE / 256];
#pragma unroll
        for (int i = 0; i < CH_TILE / 256; ++i) acc[i] = mk<T>(0, 0);
        if (n0 >= D) {
            for (int t = 0; t < nnz; ++t) {
                const cx<T> w = hv[t];
                const cx<T>* sp = cur + threadIdx.x - hd[t];
#pragma unroll
                for (int i = 0; i < CH_TILE / 256; ++i) acc[i] = cmac(acc[i], sp[256 * i], w);
            }
        } else {
            for (int t = 0; t < nnz; ++t) {
                const int d = hd[t];
                const cx<T> w = hv[t];
                const cx<T>* sp = cur + threadIdx.x - d;
#pragma unroll
                for (int i = 0; i < CH_TILE / 256; ++i)
                    if ((int64_t)d <= n0 + threadIdx.x + 256 * i) acc[i] = cmac(acc[i], sp[256 * i], w);
            }
        }
        cx<T>* op = out + b * L + n0 + threadIdx.x;
        if (whole) {
#pragma unroll
            for (int i = 0; i < CH_TILE / 256; ++i) op[256 * i] = acc[i];
        } else {
#pragma unroll
            for (int i = 0; i < CH_TILE / 256; ++i)
                if (n0 + threadIdx.x + 256 * i < L) op[256 * i] = acc[i];
        }
        __syncthreads();
        for (int j = threadIdx.x; j < D - 1; j += 256) sn[j] = sn[CH_TILE + j];     // D - 1 <= CH_TILE: source and destination are disjoint
        __syncthreads();
    }
}

// sum |x|^2 per stream in double (first half of `Noise.m:3`); also used by ofdm_tx_chain_p for the shapes its fast kernel does not cover
int ofdm_stream_power_sum(ofdm_ctx* ctx, const void* in, int64_t B, int64_t L, double* psum) {
    if (B * L == 0) { CUDA_TRY(ctx, cudaMemsetAsync(psum, 0, sizeof(double) * B, ctx->stream)); return OFDM_OK; }
    const int bx = (int)std::min<int64_t>(cdiv64(L, 256 * 8), POWER_MAX_BLOCKS);
    double* partial = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync((void**)&partial, sizeof(double) * (size_t)B * bx, ctx->stream));
    DISPATCH_T(ctx, { stream_power_kernel<T><<<dim3((unsigned)B, bx), 256, 0, ctx->stream>>>((const cx<T>*)in, L, partial); });
    ctx->launches++;
    stream_power_finish_kernel<<<(unsigned)cdiv64(B, 256), 256, 0, ctx->stream>>>(partial, B, bx, psum);
    LAUNCH_CHECK(ctx);
    cudaFreeAsync(partial, ctx->stream);
    return OFDM_OK;
}

int ofdm_power_finish(ofdm_ctx* ctx, const double* partial, int64_t B, int nb, double* power_sum) {     // power_sum[b] = partial[b][0] + ... in order
    if (B == 0) return OFDM_OK;
    stream_power_finish_kernel<<<(unsigned)cdiv64(B, 256), 256, 0, ctx->stream>>>(partial, B, nb, power_sum);
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// Shared launcher of the fused channel kernel.  nsto / cfo NULL: Task-5 order (noise, multipath); both given: Task-4 order.
static int channel_fused_launch(ofdm_ctx* ctx, const void* tx, int64_t B, int64_t L, const double* snr_db, const double* power_sum, const void* normals,
                                uint64_t seed, int64_t first_stream_id, const int32_t* nsto, const double* cfo, int Nfft, const void* h, int D, void* rx) {
    // scratch: power sums | sigma | compacted taps | their delays | tap count
    const size_t o_sig = sizeof(double) * (size_t)B, o_hv = o_sig + sizeof(double) * (size_t)B, o_hd = o_hv + sizeof(double2) * (size_t)D,
                 o_nnz = o_hd + sizeof(int) * (size_t)((D + 3) & ~3);
    char* scr = (char*)ctx_scratch(ctx, o_nnz + 16);
    REQUIRE(ctx, scr != nullptr, "scratch allocation failed");
    const double* psum = power_sum;
    if (!psum) {                                  // no power handed over by the TX stage: one extra pass over the signal
        int rc = ofdm_stream_power_sum(ctx, tx, B, L, (double*)scr);
        if (rc) return rc;
        psum = (const double*)scr;
    }
    const bool imp = nsto != nullptr;
    DISPATCH_T(ctx, {
        channel_prep_kernel<T><<<(unsigned)cdiv64(B, 256), 256, 0, ctx->stream>>>(B, L, snr_db, psum, (const cx<T>*)h, D, (T*)(scr + o_sig), (cx<T>*)(scr + o_hv),
                                                                                 (int*)(scr + o_hd), (int*)(scr + o_nnz));
        ctx->launches++;
        const size_t smem = sizeof(cx<T>) * (size_t)(CH_TILE + 2 * D - 1) + sizeof(int) * (size_t)D;
        auto k = imp ? channel_t5_kernel<T, true> : channel_t5_kernel<T, false>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<dim3((unsigned)B, (unsigned)cdiv64(L, (int64_t)CH_TILE * CH_CHUNK)), 256, smem, ctx->stream>>>((const cx<T>*)tx, L, (const T*)(scr + o_sig), (const T*)normals, seed,
                                                                                         first_stream_id, (const cx<T>*)(scr + o_hv), (const int*)(scr + o_hd),
                                                                                         (const int*)(scr + o_nnz), D, (cx<T>*)rx, nsto, cfo, imp ? 1.0 / Nfft : 0.0);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_channel_t4_p(ofdm_ctx* ctx, const void* tx, int64_t B, int64_t L, const double* snr_db, const double* power_sum, const void* normals,
                                 uint64_t seed, int64_t first_stream_id, const int32_t* nsto, const double* cfo, int Nfft, const void* h, int D, void* rx) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, tx && rx && snr_db && nsto && cfo && h && B >= 0 && L >= 0 && Nfft > 0 && tx != rx, "bad argument (in-place not supported)");
    REQUIRE(ctx, D >= 1 && D <= CH_MAXD, "impulse response of 1..1024 samples");
    if (B * L == 0) return OFDM_OK;
    return channel_fused_launch(ctx, tx, B, L, snr_db, power_sum, normals, seed, first_stream_id, nsto, cfo, Nfft, h, D, rx);
}

extern "C" int ofdm_channel_t5(ofdm_ctx* ctx, const void* tx, int64_t B, int64_t L, const double* snr_db, const void* normals,
                               uint64_t seed, int64_t first_stream_id, const void* h, int D, void* rx) {
    return ofdm_channel_t5_p(ctx, tx, B, L, snr_db, nullptr, normals, seed, first_stream_id, h, D, rx);
}
extern "C" int ofdm_channel_t5_p(ofdm_ctx* ctx, const void* tx, int64_t B, int64_t L, const double* snr_db, const double* power_sum, const void* normals,
                                 uint64_t seed, int64_t first_stream_id, const void* h, int D, void* rx) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, tx && rx && B >= 0 && L >= 0, "bad argument");
    if (B * L == 0) return OFDM_OK;
    size_t esz = ctx->precision == OFDM_PREC_F64 ? sizeof(double2) : sizeof(float2);
    if (snr_db && h && D >= 1 && D <= CH_MAXD && tx != rx)
        return channel_fused_launch(ctx, tx, B, L, snr_db, power_sum, normals, seed, first_stream_id, nullptr, nullptr, 0, h, D, rx);
    if (snr_db && h) {
        // noise must precede the filter; stage the noisy stream in a second buffer region
        void* tmp = nullptr;
        CUDA_TRY(ctx, cudaMallocAsync(&tmp, esz * B * L, ctx->stream));
        int rc = ofdm_add_noise(ctx, tx, B, L, snr_db, normals, seed, first_stream_id, tmp, nullptr);
        if (!rc) rc = ofdm_apply_fir(ctx, tmp, B, L, h, D, 0, rx);
        cudaFreeAsync(tmp, ctx->stream);
        return rc;
    }
    if (snr_db) return ofdm_add_noise(ctx, tx, B, L, snr_db, normals, seed, first_stream_id, rx, nullptr);
    if (h) return ofdm_apply_fir(ctx, tx, B, L, h, D, 0, rx);
    CUDA_TRY(ctx, cudaMemcpyAsync(rx, tx, esz * B * L, cudaMemcpyDeviceToDevice, ctx->stream));
    return OFDM_OK;
}

// ---- static tapped-delay-line fading channel (stands in for `lteFadingChannel`, `Task 5/Task5_part2.m:27-34,152-154`)
// The reference draws one static realisation per Monte-Carlo run (DopplerFreq = 0, InitPhase "Random", per-run Seed)
// of the LTE EPA / EVA / ETU profile at SamplingRate 4e7 and obtains its impulse response by filtering a unit
// impulse.  LTE Toolbox source is not available, so this is the PUBLISHED model only -- 3GPP TS 36.101 Annex B.2.1
// tap delays and relative powers, Rayleigh tap gains normalised to unit total average power, fractional delays by
// a Hann-windowed sinc interpolator with a fixed lead of TDL_LEAD samples -- and its draws do not reproduce
// MATLAB's (parity unpinned; imported taps go through ofdm_apply_fir directly).
#define TDL_LEAD 7
#define TDL_MAXP 9
struct TdlProfile { int n; double delay_ns[TDL_MAXP]; double power_db[TDL_MAXP]; };
static const TdlProfile TDL_TABLE[3] = {
    {7, {0, 30, 70, 90, 110, 190, 410, 0, 0}, {0.0, -1.0, -2.0, -3.0, -8.0, -17.2, -20.8, 0, 0}},                       // EPA
    {9, {0, 30, 150, 310, 370, 710, 1090, 1730, 2510}, {0.0, -1.5, -1.4, -3.6, -0.6, -9.1, -7.0, -12.0, -16.9}},       // EVA
    {9, {0, 50, 120, 200, 230, 500, 1600, 2300, 5000}, {-1.0, -1.0, -1.0, 0.0, 0.0, 0.0, -3.0, -5.0, -7.0}}};          // ETU
struct TdlDev { int n; float delay[TDL_MAXP]; float amp[TDL_MAXP]; };

extern "C" int ofdm_tdl_info(int profile, double fs_hz, int* n_paths, int* h_len, double* delays_samples) {
    if (profile < 0 || profile > 2 || !(fs_hz > 0)) return OFDM_ERR_INVALID;
    const TdlProfile& t = TDL_TABLE[profile];
    double dmax = 0;
    for (int i = 0; i < t.n; ++i) { double d = t.delay_ns[i] * 1e-9 * fs_hz; if (delays_samples) delays_samples[i] = d; dmax = std::max(dmax, d); }
    if (n_paths) *n_paths = t.n;
    if (h_len) *h_len = (int)ceil(dmax) + 2 * TDL_LEAD + 1;
    return OFDM_OK;
}

// one thread per (stream, tap of the impulse response): h[n] = sum_p g_p * w(n - LEAD - d_p), w = Hann-windowed sinc of half width LEAD
template <typename T>
__global__ void tdl_kernel(TdlDev t, int64_t B, int Lh, uint64_t seed, int64_t first_stream, cx<T>* __restrict__ h, cx<T>* __restrict__ gains) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * Lh) return;
    const int64_t b = i / Lh;
    const int n = (int)(i - b * Lh);
    float ar = 0.f, ai = 0.f;
    for (int p = 0; p < t.n; ++p) {
        float g1, g2;
        philox_normal_pair(seed ^ 0x74646c5f63686e6cULL, (uint64_t)(first_stream + b), (uint64_t)p, g1, g2);   // own key space ("tdl_chnl")
        const float gr = t.amp[p] * g1 * 0.70710678118654752f, gi = t.amp[p] * g2 * 0.70710678118654752f;
        if (n == 0 && gains) gains[b * t.n + p] = mk<T>((T)gr, (T)gi);
        const float x = (float)n - (float)TDL_LEAD - t.delay[p];
        float w = 0.f;
        if (fabsf(x) < (float)TDL_LEAD) {
            const float sinc = (x == 0.f) ? 1.f : sinpif(x) / (3.14159265358979323846f * x);
            w = sinc * (0.5f + 0.5f * cospif(x / (float)TDL_LEAD));
        }
        ar += gr * w; ai += gi * w;
    }
    h[i] = mk<T>((T)ar, (T)ai);
}
extern "C" int ofdm_tdl_channel(ofdm_ctx* ctx, int profile, double fs_hz, int64_t B, uint64_t seed, int64_t first_stream_id, int h_len,
                                void* h_dev, void* gains_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    int np = 0, need = 0;
    REQUIRE(ctx, ofdm_tdl_info(profile, fs_hz, &np, &need, nullptr) == OFDM_OK, "unknown delay profile or sampling rate");
    REQUIRE(ctx, h_dev && B >= 0 && h_len >= need, "h_dev missing or shorter than ofdm_tdl_info's h_len");
    if (B == 0) return OFDM_OK;
    const TdlProfile& t = TDL_TABLE[profile];
    TdlDev d;
    d.n = t.n;
    double ptot = 0;
    for (int i = 0; i < t.n; ++i) ptot += pow(10.0, t.power_db[i] / 10.0);
    for (int i = 0; i < TDL_MAXP; ++i) {
        d.delay[i] = i < t.n ? (float)(t.delay_ns[i] * 1e-9 * fs_hz) : 0.f;
        d.amp[i] = i < t.n ? (float)sqrt(pow(10.0, t.power_db[i] / 10.0) / ptot) : 0.f;
    }
    DISPATCH_T(ctx, { tdl_kernel<T><<<(unsigned)cdiv64(B * h_len, 128), 128, 0, ctx->stream>>>(d, B, h_len, seed, first_stream_id, (cx<T>*)h_dev, (cx<T>*)gains_dev); });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- channel-estimate error of `Task5_part2.m:200-203`: (H - Hest)(H - Hest)' / N per stream, accumulated in double
template <typename T>
__global__ void mse_kernel(const cx<T>* __restrict__ a, int64_t a_stride, const cx<T>* __restrict__ bb, int64_t b_stride, int n, double* __restrict__ out) {
    __shared__ double red[32];
    const int64_t s = blockIdx.x;
    double acc = 0;
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
        const cx<T> x = a[s * a_stride + k], y = bb[s * b_stride + k];
        const double dr = (double)x.x - (double)y.x, di = (double)x.y - (double)y.y;
        acc += dr * dr + di * di;
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) out[s] = acc / (double)n;
}
extern "C" int ofdm_mse(ofdm_ctx* ctx, const void* a_dev, int64_t a_stride, const void* b_dev, int64_t b_stride, int64_t B, int n, double* out_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, a_dev && b_dev && out_dev && B >= 0 && n > 0 && a_stride >= n && b_stride >= n, "bad argument");
    if (B == 0) return OFDM_OK;
    DISPATCH_T(ctx, { mse_kernel<T><<<(unsigned)B, 256, 0, ctx->stream>>>((const cx<T>*)a_dev, a_stride, (const cx<T>*)b_dev, b_stride, n, out_dev); });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}
// Same kernel against ONE reference row shared by the batch (a_stride 0; not exported): ofdm_sweep_mse compares every estimate
// with the single true response.  Per stream the sums are those of ofdm_mse on a replicated reference, bit for bit.
int ofdm_mse_shared_ref(ofdm_ctx* ctx, const void* ref_dev, const void* b_dev, int64_t b_stride, int64_t B, int n, double* out_dev) {
    REQUIRE(ctx, ref_dev && b_dev && out_dev && B >= 0 && n > 0 && b_stride >= n, "bad argument");
    if (B == 0) return OFDM_OK;
    DISPATCH_T(ctx, { mse_kernel<T><<<(unsigned)B, 256, 0, ctx->stream>>>((const cx<T>*)ref_dev, 0, (const cx<T>*)b_dev, b_stride, n, out_dev); });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}
