// OFDM_map_carriers / OFDM_modulator / OFDM_demodulator / get_payload / plain FFT (generic sizes).
#include "fft.cuh"

// ---- OFDM_map_carriers (`Task 5/OFDM_map_carriers.m:2-8`).  slot[k]: >=0 data rank, -1-p pilot
// row p, INT_MIN unused.  Pilot assignment comes second in the reference, so pilots win overlaps.
#define SLOT_ZERO (-2147483647 - 1)
template <typename T>
__global__ void map_carriers_kernel(const cx<T>* __restrict__ qam, int64_t B, int S, int Nfft, int Nd,
                                    const int32_t* __restrict__ slot, const cx<T>* __restrict__ pilots /* Np x S col-major, or 1 */,
                                    int pilot_stride /* Np, or 0 for scalar */, cx<T>* __restrict__ grid) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t n = B * S * (int64_t)Nfft;
    if (i >= n) return;
    int k = (int)(i % Nfft);
    int64_t bs = i / Nfft;
    int s = (int)(bs % S);
    int64_t b = bs / S;
    int sl = slot[k];
    cx<T> v = mk<T>(0, 0);
    if (sl >= 0) v = qam[(b * S + s) * (int64_t)Nd + sl];           // data(d, s) = QAM(s*Nd + d)
    else if (sl != SLOT_ZERO) { int p = -1 - sl; v = pilot_stride ? pilots[(int64_t)s * pilot_stride + p] : pilots[0]; }
    grid[i] = v;
}

static int build_slots(ofdm_ctx* ctx, int Nfft, const int32_t* data, int Nd, const int32_t* pil, int Np, std::vector<int32_t>& slot) {
    slot.assign(Nfft, SLOT_ZERO);
    for (int d = 0; d < Nd; ++d) { if (data[d] < 1 || data[d] > Nfft) return ctx_fail(ctx, OFDM_ERR_INVALID, "data carrier index out of range"); slot[data[d] - 1] = d; }
    for (int p = 0; p < Np; ++p) { if (pil[p] < 1 || pil[p] > Nfft) return ctx_fail(ctx, OFDM_ERR_INVALID, "pilot carrier index out of range"); slot[pil[p] - 1] = -1 - p; }
    return OFDM_OK;
}

// pilot values (complex doubles, host) -> device array of the context's type, cached
static const void* upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex) {
    if (ctx->precision == OFDM_PREC_F64) return ctx_blob(ctx, pv, n_complex * 2 * sizeof(double));
    std::vector<float> f(n_complex * 2);
    for (size_t i = 0; i < n_complex * 2; ++i) f[i] = (float)pv[i];
    return ctx_blob(ctx, f.data(), f.size() * sizeof(float));
}
const void* ofdm_upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex) { return upload_pilots(ctx, pv, n_complex); }

extern "C" int ofdm_map_carriers(ofdm_ctx* ctx, const void* qam, int64_t B, int S, int Nfft, const int32_t* data, int Nd,
                                 const int32_t* pil, int Np, const double* pv, int pilot_mode, void* grid) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && B >= 0 && S > 0 && Nfft > 0 && Nd >= 0 && Np >= 0, "bad argument");
    REQUIRE(ctx, (Nd == 0 || (qam && data)) && (Np == 0 || (pil && pv)), "null pointer");
    if (B == 0) return OFDM_OK;
    std::vector<int32_t> slot;
    int rc = build_slots(ctx, Nfft, data, Nd, pil, Np, slot);
    if (rc) return rc;
    const int32_t* slot_d = (const int32_t*)ctx_blob(ctx, slot.data(), slot.size() * sizeof(int32_t));
    const void* pil_d = nullptr;
    int stride = 0;
    std::vector<double> tmp;
    if (Np > 0) {
        if (pilot_mode == 0) { pil_d = upload_pilots(ctx, pv, (size_t)Np * S); stride = Np; }
        else if (pilot_mode == 1) { pil_d = upload_pilots(ctx, pv, 1); stride = 0; }
        else if (pilot_mode == 2) {  // v1 (`Task 1/OFDM_map_carriers.m:7-11`): +a, a*exp(i*pi), conj by the ctranspose
            tmp.resize((size_t)Np * S * 2);
            for (int s = 0; s < S; ++s)
                for (int p = 0; p < Np; ++p) {
                    double re = (p & 1) ? pv[0] * cos(M_PI) : pv[0], im = (p & 1) ? -(pv[0] * sin(M_PI)) : 0.0;
                    tmp[((size_t)s * Np + p) * 2] = re; tmp[((size_t)s * Np + p) * 2 + 1] = im;
                }
            pil_d = upload_pilots(ctx, tmp.data(), (size_t)Np * S); stride = Np;
        } else return ctx_fail(ctx, OFDM_ERR_INVALID, "pilot_mode must be 0, 1 or 2");
        REQUIRE(ctx, pil_d != nullptr, "device upload failed");
    }
    REQUIRE(ctx, slot_d != nullptr, "device upload failed");
    int64_t n = B * S * (int64_t)Nfft;
    DISPATCH_T(ctx, {
        map_carriers_kernel<T><<<(unsigned)cdiv64(n, 256), 256, 0, ctx->stream>>>((const cx<T>*)qam, B, S, Nfft, Nd, slot_d, (const cx<T>*)pil_d, stride, (cx<T>*)grid);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- get_payload (`Task 5/get_payload.m:2-4`)
template <typename T>
__global__ void get_payload_kernel(const cx<T>* __restrict__ grid, int64_t BS, int Nfft, int Nd, const int32_t* __restrict__ data0,
                                   cx<T>* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= BS * Nd) return;
    int d = (int)(i % Nd);
    int64_t bs = i / Nd;
    out[i] = grid[bs * Nfft + data0[d]];
}
extern "C" int ofdm_get_payload(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, const int32_t* data, int Nd, void* out) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && out && data && B >= 0 && S > 0 && Nd > 0, "bad argument");
    if (B == 0) return OFDM_OK;
    std::vector<int32_t> d0(Nd);
    for (int d = 0; d < Nd; ++d) { REQUIRE(ctx, data[d] >= 1 && data[d] <= Nfft, "carrier index out of range"); d0[d] = data[d] - 1; }
    const int32_t* dd = (const int32_t*)ctx_blob(ctx, d0.data(), d0.size() * sizeof(int32_t));
    REQUIRE(ctx, dd != nullptr, "device upload failed");
    int64_t n = B * S * (int64_t)Nd;
    DISPATCH_T(ctx, {
        get_payload_kernel<T><<<(unsigned)cdiv64(n, 256), 256, 0, ctx->stream>>>((const cx<T>*)grid, B * S, Nfft, Nd, dd, (cx<T>*)out);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ---- generic FFT kernel: one block per transform.
// MODE 0 plain, 1 OFDM_modulator (IFFT, 1/N, CP prepend), 2 OFDM_demodulator (CP strip, FFT).
template <typename T, int MODE, bool INV>
__global__ void fft_kernel(const cx<T>* __restrict__ in, cx<T>* __restrict__ out, int N, int logN, int Tg,
                           const cx<T>* __restrict__ tw) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using C = cx<T>;
    C* a = (C*)smem_raw;
    C* b = a + N;
    const int64_t blk = blockIdx.x;
    const C* src = (MODE == 2) ? in + blk * (int64_t)(N + Tg) + Tg : in + blk * (int64_t)N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) a[i] = src[i];
    __syncthreads();
    C* r = block_fft<T, INV>(a, b, N, logN, tw);
    const T scale = INV ? (T)1 / (T)N : (T)1;
    if (MODE == 1) {
        C* dst = out + blk * (int64_t)(N + Tg);
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            C v = cscale(r[i], scale);
            dst[Tg + i] = v;
            if (i >= N - Tg) dst[i - (N - Tg)] = v;   // cp = OFDM_time(end-T_guard+1:end,:)
        }
    } else {
        C* dst = out + blk * (int64_t)N;
        for (int i = threadIdx.x; i < N; i += blockDim.x) dst[i] = INV ? cscale(r[i], scale) : r[i];
    }
}

template <typename T, int MODE, bool INV>
static int launch_fft(ofdm_ctx* ctx, const void* in, void* out, int64_t n_batch, int N, int Tg) {
    const void* tw = ctx_twiddles(ctx, N);
    if (!tw) return ctx_fail(ctx, OFDM_ERR_CUDA, "twiddle table allocation failed");
    size_t smem = 2 * (size_t)N * sizeof(cx<T>);
    auto kern = fft_kernel<T, MODE, INV>;
    if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)kern, (int)smem));
    int64_t done = 0;
    while (done < n_batch) {  // gridDim.x limit is 2^31-1; chunk anyway
        int64_t nb = std::min<int64_t>(n_batch - done, 1 << 30);
        const cx<T>* src = (const cx<T>*)in + done * (int64_t)(MODE == 2 ? N + Tg : N);
        cx<T>* dst = (cx<T>*)out + done * (int64_t)(MODE == 1 ? N + Tg : N);
        kern<<<(unsigned)nb, fft_threads(N), smem, ctx->stream>>>(src, dst, N, ilog2(N), Tg, (const cx<T>*)tw);
        LAUNCH_CHECK(ctx);
        done += nb;
    }
    return OFDM_OK;
}

static int check_fft_size(ofdm_ctx* ctx, int N) {
    if (!is_pow2(N) || N < 2) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "FFT size must be a power of two (got %d)", N);
    int maxN = ctx->precision == OFDM_PREC_F64 ? 4096 : 8192;
    if (N > maxN) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "FFT size %d exceeds the shared-memory kernel limit %d", N, maxN);
    return OFDM_OK;
}

extern "C" int ofdm_fft(ofdm_ctx* ctx, const void* in, void* out, int64_t n_batch, int N, int inverse) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, in && out && n_batch >= 0, "bad argument");
    int rc = check_fft_size(ctx, N);
    if (rc) return rc;
    if (n_batch == 0) return OFDM_OK;
    DISPATCH_T(ctx, { return inverse ? launch_fft<T, 0, true>(ctx, in, out, n_batch, N, 0) : launch_fft<T, 0, false>(ctx, in, out, n_batch, N, 0); });
}
extern "C" int ofdm_modulate(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, int Tg, void* time) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && time && B >= 0 && S > 0 && Tg >= 0 && Tg <= Nfft, "bad argument");
    int rc = check_fft_size(ctx, Nfft);
    if (rc) return rc;
    if (B == 0) return OFDM_OK;
    DISPATCH_T(ctx, { return launch_fft<T, 1, true>(ctx, grid, time, B * S, Nfft, Tg); });
}
extern "C" int ofdm_demodulate(ofdm_ctx* ctx, const void* time, int64_t B, int S, int Nfft, int Tg, void* grid) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && time && B >= 0 && S > 0 && Tg >= 0, "bad argument");
    int rc = check_fft_size(ctx, Nfft);
    if (rc) return rc;
    if (B == 0) return OFDM_OK;
    DISPATCH_T(ctx, { return launch_fft<T, 2, false>(ctx, time, grid, B * S, Nfft, Tg); });
}
