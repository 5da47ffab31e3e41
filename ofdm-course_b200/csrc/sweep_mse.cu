// ofdm_sweep_mse: the Task-5 channel-estimation study over SNR as ONE library call per rank.
//
// Replaces the MSE half of the SNR loop `Task 5/Main_model_Task_5.m:303-346`: at every SNR point Noise -> multipath ->
// OFDM_demodulator -> LS_CE / MMSE_CE / MP_estimate / OMP_estimate, and the MSE of each estimate against the true
// frequency response (`:195-205`).  Work decomposition, stream numbering and Philox keys are those of ofdm_sweep_ber
// (sweep.cu): global stream g = snr_index * streams_per_point + j, rank r of `world` takes the contiguous share of
// ofdm_sweep_share, tiles never straddle an SNR point, temporaries are stream-ordered and reused by every tile.
//
// Every estimator reads symbol 1 only (`LS_CE.m:27-28`, `MMSE_CE.m:17`, `Main_model_Task_5.m:191`), so the channel and
// the demodulator are not run over the whole stream: mse_front_end_kernel forms exactly the noisy samples that feed
// symbol 1's useful part, filters them, takes the FFT and writes the measurement vector y = RX(pilot_loc,1)./Xp -- bit
// for bit what ofdm_channel_t5_p -> ofdm_demodulate -> ofdm_pilot_ls give on the same stream.  Everything after it is an
// existing kernel on y: interpolate (LS_CE), ifft (`:179`), the MMSE_CE kernel on measurement vectors, MP / Batch-OMP on
// the partial-DFT descriptor, and the per-stream MSE.  Each (point, estimator, stream) cell is written by exactly one
// call, so the caller's sum over ranks is exact and no floating-point atomics are involved.
#include "fft.cuh"
#include "philox.cuh"
#include "pursuit_common.cuh"
#include "sweep_common.cuh"

int ofdm_stream_power_sum(ofdm_ctx* ctx, const void* in, int64_t B, int64_t L, double* power_sum);
int ofdm_mmse_ce_meas(ofdm_ctx* ctx, const void* y, int64_t B, const int32_t* loc, int Np, int Nc, const void* h, int h_len, const double* snr_db,
                      void* H);
int ofdm_mse_shared_ref(ofdm_ctx* ctx, const void* ref_dev, const void* b_dev, int64_t b_stride, int64_t B, int n, double* out_dev);
const void* ofdm_upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex);

#define FE_THREADS 256

// One CTA per stream.  Slot j of `sn` holds the noisy sample Tg - (D-1) + j, so sn covers the D - 1 samples of FIR history
// before symbol 1's useful part and the Nfft samples of it; the FIR output goes to `fa`, and the FFT ping-pongs between fa
// and sn.  The operations are those of channel_t5_kernel (noise x + sigma*g with the pair's Philox quad, cmac over the
// non-zero taps in ascending delay, samples before the stream start absent), fft_kernel (MODE 2) and pilot_ls_kernel.
template <typename T>
__global__ void __launch_bounds__(FE_THREADS) mse_front_end_kernel(const cx<T>* __restrict__ tx, int64_t tx_stride,
                                                                   const T* __restrict__ sigma_g, uint64_t seed, int64_t first_stream, const cx<T>* __restrict__ hv_g,
                                                                   const int* __restrict__ hd_g, int nnz, int D, int Nfft, int logN, int Tg,
                                                                   const cx<T>* __restrict__ tw, const int32_t* __restrict__ loc0,
                                                                   const cx<T>* __restrict__ xp, int Np, cx<T>* __restrict__ y) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* sn = (cx<T>*)smem_raw;
    cx<T>* fa = sn + Nfft + D - 1;
    cx<T>* hv = fa + Nfft;
    int* hd = (int*)(hv + nnz);
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x;
    for (int t = tid; t < nnz; t += FE_THREADS) { hv[t] = hv_g[t]; hd[t] = hd_g[t]; }
    const T sigma = sigma_g[b];
    const cx<T>* x = tx + b * tx_stride;
    const uint64_t sid = (uint64_t)(first_stream + b);
    const int base = Tg - (D - 1);                               // sample held by slot 0 (symbol 1 lies in the first 16k samples)
    const int lo = base > 0 ? base : 0, hi = Tg + Nfft;
    for (int pr = (lo >> 1) + tid; 2 * pr < hi; pr += FE_THREADS) {
        float g[4];
        philox_normal_quad(seed, sid, (uint64_t)pr, g);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int n = 2 * pr + e;
            if (n >= lo && n < hi) { const cx<T> v = x[n]; sn[n - base] = mk<T>(v.x + sigma * (T)g[2 * e], v.y + sigma * (T)g[2 * e + 1]); }
        }
    }
    __syncthreads();
    for (int k = tid; k < Nfft; k += FE_THREADS) {
        const int n = Tg + k;
        cx<T> acc = mk<T>(0, 0);
        for (int t = 0; t < nnz; ++t) {
            const int d = hd[t];
            if (d <= n) acc = cmac(acc, sn[k + (D - 1) - d], hv[t]);
        }
        fa[k] = acc;
    }
    __syncthreads();
    const cx<T>* r = block_fft<T, false>(fa, sn, Nfft, logN, tw);
    for (int q = tid; q < Np; q += FE_THREADS) y[b * Np + q] = cdiv(r[loc0[q]], xp[q]);
}

// Per stream of a tile: the SNR the MMSE kernel reads, and sigma from the power of the WHOLE stream and its full length
// (`Noise.m:3-5`), formed as channel_prep_kernel forms it.
template <typename T>
__global__ void mse_prep_kernel(int64_t n, int64_t L, double snr_db, const double* __restrict__ power_sum, int64_t ps_stride, double* __restrict__ snr,
                                T* __restrict__ sigma) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const double P = power_sum[b * ps_stride] / (double)L;
    snr[b] = snr_db;
    sigma[b] = (T)sqrt(P / pow(10.0, snr_db / 10.0) / 2);
}

// row[0] += streams of the tile, row[1] += OMP frames with at least one near-tie iteration (one CTA, integer sums)
__global__ void mse_counts_kernel(const int32_t* __restrict__ near, int64_t n, int64_t* __restrict__ row) {
    __shared__ int red[32];
    int v = 0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) v += near[i] != 0;
    v = block_sum(v, red);
    if (threadIdx.x == 0) { row[0] += n; row[1] += v; }
}

extern "C" int ofdm_sweep_mse(ofdm_ctx* ctx, const ofdm_link_params* lp, const ofdm_sweep_params* sp, int Ldict, double* mse_dev, int64_t* counts_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, lp && sp && mse_dev && counts_dev, "null pointer");
    REQUIRE(ctx, sp->chain == OFDM_SWEEP_TASK5, "the MSE sweep runs the Task-5 chain (chain must be OFDM_SWEEP_TASK5)");
    REQUIRE(ctx, sp->n_snr > 0 && sp->snr_db_host && sp->streams_per_point > 0, "need at least one SNR point and one stream per point");
    REQUIRE(ctx, sp->world > 0 && sp->rank >= 0 && sp->rank < sp->world, "bad rank / world");
    REQUIRE(ctx, sp->n_taps >= 1 && sp->taps_host, "the MSE sweep needs a multipath channel (n_taps >= 1; K = n_taps)");
    REQUIRE(ctx, sp->n_taps <= PU_MAXK, "K = n_taps must be at most 32");
    const int Nfft = lp->Nfft, Tg = lp->Tg, Nc = lp->N_carrier, Np = lp->Np, S = lp->S, K = sp->n_taps;
    const bool f64 = ctx->precision == OFDM_PREC_F64;
    REQUIRE(ctx, is_pow2(Nfft) && Nfft >= 8 && Nfft <= (f64 ? 4096 : 8192), "Nfft must be a power of two in 8..8192 (8..4096 in FP64)");
    REQUIRE(ctx, S >= 1 && Tg >= 0 && Tg <= Nfft, "bad symbol count or guard length");
    REQUIRE(ctx, is_pow2(Nc) && Nc >= 2 && Nc <= Nfft, "N_carrier must be a power of two (h = ifft(H_LS) runs on the block FFT) and <= Nfft");
    REQUIRE(ctx, Np >= 2 && lp->pilot_carriers_host && lp->pilot_vals_host, "need at least two pilots");
    for (int q = 0; q < Np; ++q)
        REQUIRE(ctx, lp->pilot_carriers_host[q] >= 1 && lp->pilot_carriers_host[q] <= Nc && (q == 0 || lp->pilot_carriers_host[q] > lp->pilot_carriers_host[q - 1]),
                "pilot carriers must be strictly increasing within 1..N_carrier");
    REQUIRE(ctx, Ldict >= Np, "Ldict must be >= Np (MP_estimate searches the first Np columns)");
    REQUIRE(ctx, Ldict <= Nfft, "Ldict must be <= Nfft");
    REQUIRE(ctx, lp->Nd >= 0 && (lp->Nd == 0 || lp->data_carriers_host), "bad data-carrier list");
    std::vector<double> h;                                    // later rows overwrite, as `get_MP_channel_resp.m:14`
    REQUIRE(ctx, sweep_dense_taps(sp->taps_host, K, Nfft, h), "tap delays must be integers in [0, Nfft)");
    const int D = (int)h.size();
    const int64_t L = (int64_t)S * (Nfft + Tg);
    const size_t esz = f64 ? sizeof(double2) : sizeof(float2);
    int64_t words = 0;
    if (lp->Nd > 0) {
        ConstTable ct = host_constellation(lp->constellation);
        REQUIRE(ctx, ct.bps > 0, "unknown constellation");
        const int64_t stream_bits = (int64_t)S * lp->Nd * ct.bps;
        REQUIRE(ctx, stream_bits % 32 == 0, "the sweep needs word-aligned streams (S * Nd * bps divisible by 32)");
        words = stream_bits / 32;
    }

    // the channel's non-zero taps in ascending delay, in the context's type
    std::vector<double> hv_d;
    std::vector<float> hv_f;
    std::vector<int> hd;
    for (int d = 0; d < D; ++d) {
        if (f64 ? h[d] != 0.0 : (float)h[d] != 0.f) { hv_d.push_back(h[d]); hv_d.push_back(0.0); hv_f.push_back((float)h[d]); hv_f.push_back(0.f); hd.push_back(d); }
    }
    const int nnz = (int)hd.size();
    const void* hv_dev = nullptr;
    const int* hd_dev = nullptr;
    if (nnz) {
        hv_dev = f64 ? ctx_blob(ctx, hv_d.data(), sizeof(double) * hv_d.size()) : ctx_blob(ctx, hv_f.data(), sizeof(float) * hv_f.size());
        hd_dev = (const int*)ctx_blob(ctx, hd.data(), sizeof(int) * hd.size());
        REQUIRE(ctx, hv_dev && hd_dev, "device upload failed");
    }
    std::vector<int32_t> p0(Np);
    for (int q = 0; q < Np; ++q) p0[q] = lp->pilot_carriers_host[q] - 1;
    const int32_t* p0_dev = (const int32_t*)ctx_blob(ctx, p0.data(), sizeof(int32_t) * Np);
    const void* xp_dev = ofdm_upload_pilots(ctx, lp->pilot_vals_host, Np);      // pilotValues(:,1)
    const void* tw = ctx_twiddles(ctx, Nfft);
    REQUIRE(ctx, p0_dev && xp_dev && tw, "device upload failed");
    const size_t fe_smem = esz * (size_t)(2 * Nfft + D - 1) + (esz + sizeof(int)) * (size_t)nnz;
    REQUIRE(ctx, fe_smem <= 227 * 1024, "symbol too long for the shared-memory front end");

    const SweepTiles tiles(sp->n_snr, sp->streams_per_point, sp->rank, sp->world, sp->tile_streams, 8192);
    if (tiles.count == 0) return OFDM_OK;
    const int64_t tile = tiles.tile;

    // stream-ordered temporaries, sized for one tile and reused by every tile of the call
    const bool shared_tx = lp->Nd == 0;                       // pilots only (`Main_model_Task_5.m:24-33`): one TX stream for all
    const size_t b_d = sizeof(double) * tile, b_nc = esz * (size_t)tile * Nc;
    SweepScratch scr(ctx);
    CUDA_TRY(ctx, scr.alloc({esz * Nfft, b_d, b_d, b_d, sizeof(int32_t) * tile, esz * (size_t)tile * Np, b_nc, b_nc, b_nc, esz * (size_t)tile * Nfft,
                             esz * (size_t)L * (shared_tx ? 1 : tile), shared_tx ? esz * (size_t)S * Nfft : sizeof(uint32_t) * (size_t)words * tile}));
    void* Htrue = scr.get<void>(0);
    double* psum = scr.get<double>(1);
    double* snr_d = scr.get<double>(2);
    void* sigma = scr.get<void>(3);
    int32_t* near = scr.get<int32_t>(4);
    void* y = scr.get<void>(5);
    void* Hls = scr.get<void>(6);
    void* hls = scr.get<void>(7);
    void* Hmm = scr.get<void>(8);
    void* Hpur = scr.get<void>(9);
    void* tx = scr.get<void>(10);
    void* aux = scr.get<void>(11);                            // TX grid (pilots only) or the payload words of a tile

    int rc = OFDM_OK;
    {
        std::vector<double> hh(D);
        int hl = 0;
        rc = ofdm_mp_channel_resp(ctx, sp->taps_host, K, Nfft, hh.data(), D, &hl, Htrue);   // true response, first N_carrier bins compared
    }
    if (rc == OFDM_OK && shared_tx) {
        rc = ofdm_map_carriers(ctx, nullptr, 1, S, Nfft, nullptr, 0, lp->pilot_carriers_host, Np, lp->pilot_vals_host, 0, aux);
        if (rc == OFDM_OK) rc = ofdm_modulate(ctx, aux, 1, S, Nfft, Tg, tx);
        if (rc == OFDM_OK) rc = ofdm_stream_power_sum(ctx, tx, 1, L, psum);
    }
    ofdm_link_params lp_tx = *lp;                             // as ofdm_sweep_ber: the Philox words are mapped without the scrambler
    lp_tx.scramble = 0;
    if (rc == OFDM_OK && fe_smem > 48 * 1024) {
        cudaError_t e = f64 ? cudaFuncSetAttribute(mse_front_end_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fe_smem)
                            : cudaFuncSetAttribute(mse_front_end_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fe_smem);
        if (e != cudaSuccess) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "front-end shared-memory opt-in failed: %s", cudaGetErrorString(e));
    }

    const int64_t spp = sp->streams_per_point;
    if (rc == OFDM_OK) rc = tiles.walk([&](int64_t i, int64_t j0, int64_t g, int64_t n) {   // i: SNR point of this tile
        const double snr = sp->snr_db_host[i];
        int rc = OFDM_OK;
        if (!shared_tx) {
            rc = ofdm_payload_bits(ctx, (uint32_t*)aux, n, words, sp->seed, g);
            if (rc == OFDM_OK) rc = ofdm_tx_chain_p(ctx, &lp_tx, (const uint32_t*)aux, n, tx, psum);
            if (rc) return rc;
        }
        DISPATCH_T(ctx, {
            mse_prep_kernel<T><<<(unsigned)cdiv64(n, 256), 256, 0, ctx->stream>>>(n, L, snr, psum, shared_tx ? 0 : 1, snr_d, (T*)sigma);
            mse_front_end_kernel<T><<<(unsigned)n, FE_THREADS, fe_smem, ctx->stream>>>(
                (const cx<T>*)tx, shared_tx ? 0 : L, (const T*)sigma, sp->seed, g, (const cx<T>*)hv_dev, hd_dev, nnz, D, Nfft, ilog2(Nfft), Tg,
                (const cx<T>*)tw, p0_dev, (const cx<T>*)xp_dev, Np, (cx<T>*)y);
        });
        ctx->launches += 2;
        double* row = mse_dev + (size_t)i * 4 * spp + j0;                             // [i][e][j], e = LS, MMSE, MP, OMP
        rc = ofdm_interpolate(ctx, y, n, lp->pilot_carriers_host, Np, Nc, OFDM_INTERP_SPLINE, Hls);         // LS_CE
        if (rc == OFDM_OK) rc = ofdm_fft(ctx, Hls, hls, n, Nc, 1);                                              // h = ifft(H_LS), `:179`
        if (rc == OFDM_OK) rc = ofdm_mmse_ce_meas(ctx, y, n, lp->pilot_carriers_host, Np, Nc, hls, Nc, snr_d, Hmm);
        if (rc == OFDM_OK) rc = ofdm_mse_shared_ref(ctx, Htrue, Hls, Nc, n, Nc, row);
        if (rc == OFDM_OK) rc = ofdm_mse_shared_ref(ctx, Htrue, Hmm, Nc, n, Nc, row + spp);
        if (rc == OFDM_OK) rc = ofdm_mp(ctx, y, n, Np, nullptr, Ldict, lp->pilot_carriers_host, Nfft, K, Hpur, nullptr, nullptr);
        if (rc == OFDM_OK) rc = ofdm_mse_shared_ref(ctx, Htrue, Hpur, Nfft, n, Nc, row + 2 * spp);
        if (rc == OFDM_OK)
            rc = ofdm_omp_ex(ctx, y, n, Np, nullptr, Ldict, lp->pilot_carriers_host, Nfft, K, Hpur, nullptr, nullptr, nullptr, near, sp->near_eps);
        if (rc == OFDM_OK) rc = ofdm_mse_shared_ref(ctx, Htrue, Hpur, Nfft, n, Nc, row + 3 * spp);
        if (rc == OFDM_OK) {
            mse_counts_kernel<<<1, 256, 0, ctx->stream>>>(near, n, counts_dev + 2 * i);
            ctx->launches++;
        }
        return rc;
    });
    return scr.finish(rc, "MSE sweep launch failed");
}
