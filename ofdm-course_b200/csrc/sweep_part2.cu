// ofdm_sweep_part2: the Task-5 part-2 pilot-density study as ONE library call per rank.
//
// Replaces `Task 5/Task5_part2.m:46-321`: for every pilot layout (sweep point) k and Monte-Carlo run r, a static fading
// realisation filters the point's one noisy TX stream, and the NMSE of the LS / MMSE / MP / OMP estimates and the bit errors
// after equalising with each of them are recorded.  The keys are those of part2.run_point, the composed reference: the TX
// stream of point k carries the payload prefix unscrambled, its AWGN is Philox stream k (ofdm_add_noise, power over the whole
// stream), run r of point k fades with ofdm_tdl_channel stream k * 1,000,003 + r.  Work item g = k * mc_runs + r; rank r of
// `world` takes the contiguous share of ofdm_sweep_share, tiles never straddle a point.
//
// Two kernels of this file carry the hot path; everything between them is an existing kernel.
//  * part2_front_end_kernel (one CTA per run) forms symbol 1 of FIR(noisy stream), takes the FFT and writes the measurement
//    vector y = Y(pilots,1) ./ Xp: bit for bit ofdm_apply_fir -> ofdm_demodulate -> ofdm_pilot_ls.
//  * interpolate (LS_CE on y), the MMSE kernel on measurement vectors, MP, Batch-OMP, the FFT of the true response and the
//    per-run NMSE follow.
//  * part2_decide_kernel (one CTA per (run, symbol)) forms that symbol again from the L2-resident noisy stream -- recomputing
//    is cheaper than storing Y -- and, for each of the four estimates and each data carrier, takes cdiv(Y, H_e), the nearest
//    constellation point and its margin, and counts bit errors against the payload: exactly the errors of ofdm_equalize ->
//    ofdm_get_payload -> ofdm_demap -> ofdm_ber_count.  Rx, Y, the equalised grids and the payload IQ are never stored.
// Each (point, estimator, run) NMSE cell is written by exactly one call; counters are integer sums.  No floating-point atomics.
#include "fft.cuh"
#include "pursuit_common.cuh"
#include "sweep_common.cuh"

int ofdm_mmse_ce_meas(ofdm_ctx* ctx, const void* y, int64_t B, const int32_t* loc, int Np, int Nc, const void* h, int h_len, const double* snr_db,
                      void* H);

#define P2_THREADS 256
#define P2_RUN_KEY 1000003          // fading stream of run r of point k: k * P2_RUN_KEY + r (part2.run_point)
#define P2_DEFAULT_TILE 4096

// The non-zero taps of one impulse response in ascending delay, with fir_kernel's zero test, compacted by a block scan.
// Returns the tap count (valid in every thread, the lists are synchronised on return).
template <typename T>
__device__ __forceinline__ int p2_load_taps(const cx<T>* __restrict__ h, int D, cx<T>* hv, int* hd, int* scan_sh) {
    int nnz = 0;
    for (int base = 0; base < D; base += P2_THREADS) {
        const int i = base + threadIdx.x;
        const cx<T> t = i < D ? h[i] : mk<T>(0, 0);
        const int nz = i < D && (t.x != (T)0 || t.y != (T)0);
        const int off = block_exclusive_scan(nz, scan_sh);
        if (nz) { hv[nnz + off] = t; hd[nnz + off] = i; }
        nnz += __syncthreads_count(nz);
    }
    return nnz;
}

// FFT of the useful part of one OFDM symbol of FIR(x): the symbol starts at sample n0 of the stream x (length L).  Slot j of
// `sn` holds sample n0 - (D-1) + j, so sn covers the D - 1 samples of FIR history and the Nfft samples of the symbol; the
// FIR output goes to `fa` and the FFT ping-pongs between fa and sn.  The operations are those of fir_kernel (cmac over the
// non-zero taps in ascending delay, taps with d > n absent) and fft_kernel (MODE 2).  Returns the buffer holding the result.
template <typename T>
__device__ __forceinline__ const cx<T>* p2_symbol_fft(const cx<T>* __restrict__ x, int64_t L, int64_t n0, cx<T>* sn, cx<T>* fa, const cx<T>* hv,
                                                      const int* hd, int nnz, int D, int Nfft, int logN, const cx<T>* __restrict__ tw) {
    for (int j = threadIdx.x; j < Nfft + D - 1; j += P2_THREADS) {
        const int64_t n = n0 - (D - 1) + j;
        if (n >= 0 && n < L) sn[j] = x[n];
    }
    __syncthreads();
    for (int k = threadIdx.x; k < Nfft; k += P2_THREADS) {
        const int64_t n = n0 + k;
        cx<T> acc = mk<T>(0, 0);
        for (int t = 0; t < nnz; ++t) {
            const int d = hd[t];
            if ((int64_t)d <= n) acc = cmac(acc, sn[k + (D - 1) - d], hv[t]);
        }
        fa[k] = acc;
    }
    __syncthreads();
    return block_fft<T, false>(fa, sn, Nfft, logN, tw);
}

// dynamic shared memory of both kernels: sn (Nfft + D - 1) | fa (Nfft) | hv (D) complex, then hd (D) int
static size_t p2_smem(size_t esz, int Nfft, int D) { return esz * (size_t)(2 * Nfft + 2 * D - 1) + sizeof(int) * (size_t)D; }

// One CTA per run: y[b] = FFT(FIR_b(x))(pilots, symbol 1) ./ Xp.
template <typename T>
__global__ void __launch_bounds__(P2_THREADS) part2_front_end_kernel(const cx<T>* __restrict__ x, int64_t L, const cx<T>* __restrict__ h, int D,
                                                                     int Nfft, int logN, int Tg, const cx<T>* __restrict__ tw,
                                                                     const int32_t* __restrict__ loc0, const cx<T>* __restrict__ xp, int Np,
                                                                     cx<T>* __restrict__ y) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int scan_sh[32];
    cx<T>* sn = (cx<T>*)smem_raw;
    cx<T>* fa = sn + Nfft + D - 1;
    cx<T>* hv = fa + Nfft;
    int* hd = (int*)(hv + D);
    const int64_t b = blockIdx.x;
    const int nnz = p2_load_taps<T>(h + b * D, D, hv, hd, scan_sh);
    const cx<T>* r = p2_symbol_fft<T>(x, L, Tg, sn, fa, hv, hd, nnz, D, Nfft, logN, tw);
    for (int q = threadIdx.x; q < Np; q += P2_THREADS) y[b * Np + q] = cdiv(r[loc0[q]], xp[q]);
}

// The four channel estimates of a tile: row b of estimator e starts at H[e] + b * stride[e].
template <typename T>
struct P2Est {
    const cx<T>* H[4];
    int stride[4];
};

// One CTA per (run, symbol): equalise the symbol's data carriers with each estimate, decide, count against the payload.
// counts[e] += {bit errors, -, symbols whose two smallest squared distances differ by less than near_eps}.
template <typename T>
__global__ void __launch_bounds__(P2_THREADS) part2_decide_kernel(const cx<T>* __restrict__ x, int64_t L, const cx<T>* __restrict__ h, int D,
                                                                  int Nfft, int logN, int Tg, const cx<T>* __restrict__ tw,
                                                                  const int32_t* __restrict__ dc0, int Nd, P2Est<T> est, DevConst<T> c,
                                                                  const uint32_t* __restrict__ payload, int64_t stream_bits, T near_eps,
                                                                  unsigned long long* __restrict__ counts) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int scan_sh[32];
    __shared__ int red[32];
    cx<T>* sn = (cx<T>*)smem_raw;
    cx<T>* fa = sn + Nfft + D - 1;
    cx<T>* hv = fa + Nfft;
    int* hd = (int*)(hv + D);
    const int64_t b = blockIdx.x;
    const int s = blockIdx.y;
    const int nnz = p2_load_taps<T>(h + b * D, D, hv, hd, scan_sh);
    const cx<T>* r = p2_symbol_fft<T>(x, L, (int64_t)s * (Nfft + Tg) + Tg, sn, fa, hv, hd, nnz, D, Nfft, logN, tw);
    int err[4] = {0, 0, 0, 0}, near[4] = {0, 0, 0, 0};
    const uint32_t mask = (1u << c.bps) - 1u;
    for (int m = threadIdx.x; m < Nd; m += P2_THREADS) {
        const int k = dc0[m];
        const cx<T> v = r[k];
        const uint32_t want = bits_get32(payload, ((int64_t)s * Nd + m) * c.bps, stream_bits) & mask;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const cx<T> q = cdiv(v, est.H[e][b * est.stride[e] + k]);
            T margin;
            const int idx = nearest_idx(c, q.x, q.y, &margin);
            uint32_t got = 0;                                   // bit j of the group is the MSB-first bit (bps-1-j) of idx
            for (int j = 0; j < c.bps; ++j) got |= (uint32_t)((idx >> (c.bps - 1 - j)) & 1) << j;
            err[e] += __popc(got ^ want);
            near[e] += margin < near_eps;
        }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int te = block_sum(err[e], red);
        const int tn = block_sum(near[e], red);
        if (threadIdx.x == 0) {
            if (te) atomicAdd(&counts[3 * e], (unsigned long long)te);
            if (tn) atomicAdd(&counts[3 * e + 2], (unsigned long long)tn);
        }
    }
}

// runs[0] += n, runs[1] += OMP runs with at least one near-tie iteration, counts[3 e + 1] += n * stream_bits (one CTA)
__global__ void part2_runs_kernel(const int32_t* __restrict__ near_ties, int64_t n, int64_t stream_bits, int64_t* __restrict__ runs,
                                  int64_t* __restrict__ counts) {
    __shared__ int red[32];
    int v = 0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) v += near_ties[i] != 0;
    v = block_sum(v, red);
    if (threadIdx.x == 0) {
        runs[0] += n;
        runs[1] += v;
        for (int e = 0; e < 4; ++e) counts[3 * e + 1] += n * stream_bits;
    }
}

extern "C" int ofdm_sweep_part2(ofdm_ctx* ctx, const ofdm_link_params* base, const ofdm_part2_params* pp, double* nmse_dev, int64_t* counts_dev,
                                int64_t* runs_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, base && pp && nmse_dev && counts_dev && runs_dev, "null pointer");
    REQUIRE(ctx, pp->pilot_offsets_host && pp->pilot_carriers_host && pp->ldict_host && pp->pilot_pattern_host && pp->payload_host,
            "null host array in the part-2 parameters");
    REQUIRE(ctx, pp->n_points >= 1, "need at least one sweep point (n_points >= 1)");
    const int P = pp->n_points;
    const int32_t* off = pp->pilot_offsets_host;
    REQUIRE(ctx, off[0] == 0, "pilot_offsets must start at 0");
    for (int k = 0; k < P; ++k) REQUIRE(ctx, off[k + 1] >= off[k], "pilot_offsets must be non-decreasing");
    const int Nfft = base->Nfft, Tg = base->Tg, Nc = base->N_carrier, S = base->S;
    const bool f64 = ctx->precision == OFDM_PREC_F64;
    REQUIRE(ctx, is_pow2(Nfft) && Nfft >= 8 && Nfft <= (f64 ? 4096 : 8192), "Nfft must be a power of two in 8..8192 (8..4096 in FP64)");
    REQUIRE(ctx, S >= 1 && S <= 65535 && base->SpF >= 1 && S % base->SpF == 0 && Tg >= 0 && Tg <= Nfft,
            "bad symbol count (a multiple of SpF) or guard length");
    REQUIRE(ctx, Nc >= 2 && Nc <= Nfft, "N_carrier must be in 2..Nfft");
    ConstTable ct = host_constellation(base->constellation);
    REQUIRE(ctx, ct.bps > 0, "unknown constellation");
    REQUIRE(ctx, pp->profile >= 0 && pp->profile <= 2, "profile must be 0 (EPA), 1 (EVA) or 2 (ETU)");
    int K = 0, D = 0;
    REQUIRE(ctx, ofdm_tdl_info(pp->profile, pp->fs_hz, &K, &D, nullptr) == OFDM_OK, "fs_hz must be positive");
    REQUIRE(ctx, K <= PU_MAXK, "K = n_paths must be at most 32");
    REQUIRE(ctx, D <= Nc, "the fading response (h_len of ofdm_tdl_info) must not be longer than N_carrier");
    REQUIRE(ctx, pp->mc_runs >= 1 && pp->mc_runs <= P2_RUN_KEY, "mc_runs must be in 1..1000003 (run keys k * 1000003 + r)");
    REQUIRE(ctx, pp->tile_runs >= 0, "tile_runs must be >= 0 (0 = 4096)");
    REQUIRE(ctx, pp->world > 0 && pp->rank >= 0 && pp->rank < pp->world, "bad rank / world");
    int64_t max_bits = 0;
    for (int k = 0; k < P; ++k) {
        const int32_t* pc = pp->pilot_carriers_host + off[k];
        const int Np = off[k + 1] - off[k];
        REQUIRE(ctx, Np >= 2, "every point needs at least two pilots");
        for (int q = 0; q < Np; ++q)
            REQUIRE(ctx, pc[q] >= 1 && pc[q] <= Nc && (q == 0 || pc[q] > pc[q - 1]), "pilot carriers must be strictly increasing within 1..N_carrier");
        REQUIRE(ctx, Nc - Np >= 1, "every point needs at least one data carrier (Nd >= 1)");
        REQUIRE(ctx, pp->ldict_host[k] >= Np && pp->ldict_host[k] <= Nfft, "Ldict must satisfy Np <= Ldict <= Nfft");
        max_bits = std::max<int64_t>(max_bits, (int64_t)S * (Nc - Np) * ct.bps);
    }
    REQUIRE(ctx, pp->payload_bits >= max_bits, "payload_bits is shorter than the stream of the point with the most data carriers");
    const size_t esz = f64 ? sizeof(double2) : sizeof(float2);
    const size_t smem = p2_smem(esz, Nfft, D);
    REQUIRE(ctx, smem <= 227 * 1024, "symbol plus fading response too long for the shared-memory kernels");

    const SweepTiles tiles(P, pp->mc_runs, pp->rank, pp->world, pp->tile_runs, P2_DEFAULT_TILE);
    if (tiles.count == 0) return OFDM_OK;
    const int64_t tile = tiles.tile;
    const int64_t L = (int64_t)S * (Nfft + Tg);

    // stream-ordered temporaries, sized for one tile and reused by every tile of the call
    const size_t b_sig = esz * (size_t)L, b_nc = esz * (size_t)tile * Nc, b_nf = esz * (size_t)tile * Nfft, b_idx = sizeof(int32_t) * Nc;
    SweepScratch scr(ctx);
    CUDA_TRY(ctx, scr.alloc({b_sig, b_sig, esz * (size_t)tile * D, b_nc, b_nc, b_nc, b_nc, b_nf, b_nf, b_nf, sizeof(double) * tile, sizeof(int32_t) * tile,
                             b_idx, b_idx, esz * Nc, sizeof(uint32_t) * (size_t)OFDM_BIT_WORDS(max_bits)}));
    void* tx = scr.get<void>(0);
    void* txn = scr.get<void>(1);
    void* h = scr.get<void>(2);
    void* y = scr.get<void>(3);                               // y of up to Nc pilots
    void* hpad = scr.get<void>(4);                            // true CIR zero-padded to N_carrier (the MMSE input, `:176-177`)
    void* Hls = scr.get<void>(5);
    void* Hmm = scr.get<void>(6);
    void* Hf = scr.get<void>(7);                              // fft(h zero-padded to Nfft), `:155`
    void* Hmp = scr.get<void>(8);                             // first holds h zero-padded to Nfft
    void* Homp = scr.get<void>(9);
    double* snr_d = scr.get<double>(10);
    int32_t* near = scr.get<int32_t>(11);
    // The per-point inputs that kernels read across the tiles of a point, and the SNR, live in this pool and not in the
    // context's blob cache: a call over many layouts uploads new blobs at every point (ofdm_tx_chain's tables), and the cache
    // frees a generation that is no longer requested.  Blobs fetched inside a callee are only read by its own launches.
    int32_t* p0_dev = scr.get<int32_t>(12);                   // the point's pilots, 0-based
    int32_t* dc0_dev = scr.get<int32_t>(13);                  // the point's data carriers, 0-based
    void* xp_dev = scr.get<void>(14);                         // pilotValues(:,1) in the context's type
    uint32_t* pay_dev = scr.get<uint32_t>(15);                // the point's payload prefix

    int rc = OFDM_OK;
    auto ck = [ctx](cudaError_t e) { return e == cudaSuccess ? OFDM_OK : ctx_fail(ctx, OFDM_ERR_CUDA, "part-2 sweep: %s", cudaGetErrorString(e)); };
    {                                                         // pageable H2D: the source is staged before the call returns
        std::vector<double> sv((size_t)tile, pp->snr_db);
        rc = ck(cudaMemcpyAsync(snr_d, sv.data(), sizeof(double) * tile, cudaMemcpyHostToDevice, ctx->stream));
    }
    const void* tw = ctx_twiddles(ctx, Nfft);
    if (rc == OFDM_OK && !tw) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "twiddle table allocation failed");
    if (rc == OFDM_OK && smem > 48 * 1024) {
        cudaError_t e1 = f64 ? cudaFuncSetAttribute(part2_front_end_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                             : cudaFuncSetAttribute(part2_front_end_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaError_t e2 = f64 ? cudaFuncSetAttribute(part2_decide_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                             : cudaFuncSetAttribute(part2_decide_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e1 != cudaSuccess || e2 != cudaSuccess)
            rc = ctx_fail(ctx, OFDM_ERR_CUDA, "shared-memory opt-in failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
    }

    static const uint8_t no_register[15] = {0};
    // per-point state, rebuilt when a tile starts a new point
    int cur = -1, Np = 0, Nd = 0;
    const int32_t* pc = nullptr;
    int64_t stream_bits = 0;

    if (rc == OFDM_OK) rc = tiles.walk([&](int64_t point, int64_t r0, int64_t, int64_t n) {
        const int k = (int)point;
        int rc = OFDM_OK;
        if (k != cur) {
            // the point's layout (`Task5_part2.m:50-80`): data carriers are the complement of the pilots in 1..N_carrier
            pc = pp->pilot_carriers_host + off[k];
            Np = off[k + 1] - off[k];
            Nd = Nc - Np;
            std::vector<int32_t> p0(Np), dc, dc0;
            std::vector<char> is_pilot(Nc, 0);
            for (int i = 0; i < Np; ++i) { p0[i] = pc[i] - 1; is_pilot[pc[i] - 1] = 1; }
            for (int i = 0; i < Nc; ++i)
                if (!is_pilot[i]) { dc.push_back(i + 1); dc0.push_back(i); }
            std::vector<double> pv(2 * (size_t)Np * S);           // pilot q carries pattern[q % 2] in every symbol (`:86-91`)
            for (int s = 0; s < S; ++s)
                for (int i = 0; i < Np; ++i) {
                    pv[2 * ((size_t)s * Np + i)] = pp->pilot_pattern_host[2 * (i & 1)];
                    pv[2 * ((size_t)s * Np + i) + 1] = pp->pilot_pattern_host[2 * (i & 1) + 1];
                }
            stream_bits = (int64_t)S * Nd * ct.bps;
            std::vector<uint32_t> words((size_t)OFDM_BIT_WORDS(stream_bits));   // the payload prefix, zero beyond stream_bits
            std::memcpy(words.data(), pp->payload_host, sizeof(uint32_t) * words.size());
            if (stream_bits % 32) words.back() &= (1u << (stream_bits % 32)) - 1u;
            std::vector<float> xp_f(2 * (size_t)Np);                 // pilotValues(:,1) rounded as ofdm_upload_pilots rounds it
            for (size_t i = 0; i < xp_f.size(); ++i) xp_f[i] = (float)pv[i];
            // stream-ordered after the previous point's kernels, which read the same buffers
            rc = ck(cudaMemcpyAsync(p0_dev, p0.data(), sizeof(int32_t) * Np, cudaMemcpyHostToDevice, ctx->stream));
            if (rc == OFDM_OK) rc = ck(cudaMemcpyAsync(dc0_dev, dc0.data(), sizeof(int32_t) * Nd, cudaMemcpyHostToDevice, ctx->stream));
            if (rc == OFDM_OK)
                rc = ck(f64 ? cudaMemcpyAsync(xp_dev, pv.data(), esz * Np, cudaMemcpyHostToDevice, ctx->stream)
                            : cudaMemcpyAsync(xp_dev, xp_f.data(), esz * Np, cudaMemcpyHostToDevice, ctx->stream));
            if (rc == OFDM_OK)
                rc = ck(cudaMemcpyAsync(pay_dev, words.data(), sizeof(uint32_t) * words.size(), cudaMemcpyHostToDevice, ctx->stream));
            if (rc) return rc;
            ofdm_link_params lk = *base;                             // scrambling off, as `Task5_part2.m:99-115`
            lk.Nd = Nd; lk.Np = Np;
            lk.data_carriers_host = dc.data(); lk.pilot_carriers_host = pc; lk.pilot_vals_host = pv.data();
            lk.scramble = 0;
            if (!lk.reg0_host) lk.reg0_host = no_register;           // read only when scrambling
            rc = ofdm_tx_chain(ctx, &lk, pay_dev, 1, tx);
            if (rc == OFDM_OK) rc = ofdm_add_noise(ctx, tx, 1, L, snr_d, nullptr, pp->seed, k, txn, nullptr);   // once per point, `:132`
            if (rc) return rc;
            cur = k;
        }
        rc = ofdm_tdl_channel(ctx, pp->profile, pp->fs_hz, n, pp->seed, (int64_t)k * P2_RUN_KEY + r0, D, h, nullptr);
        if (rc) return rc;
        DISPATCH_T(ctx, {
            part2_front_end_kernel<T><<<(unsigned)n, P2_THREADS, smem, ctx->stream>>>((const cx<T>*)txn, L, (const cx<T>*)h, D, Nfft, ilog2(Nfft), Tg,
                                                                                     (const cx<T>*)tw, p0_dev, (const cx<T>*)xp_dev, Np, (cx<T>*)y);
        });
        ctx->launches++;
        // h zero-padded to Nfft (-> H_f) and to N_carrier (the MMSE input)
        rc = ck(cudaMemsetAsync(Hmp, 0, esz * (size_t)n * Nfft, ctx->stream));
        if (rc == OFDM_OK) rc = ck(cudaMemsetAsync(hpad, 0, esz * (size_t)n * Nc, ctx->stream));
        if (rc == OFDM_OK) rc = ck(cudaMemcpy2DAsync(Hmp, esz * Nfft, h, esz * D, esz * D, (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
        if (rc == OFDM_OK) rc = ck(cudaMemcpy2DAsync(hpad, esz * Nc, h, esz * D, esz * D, (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
        double* row = nmse_dev + (size_t)k * 4 * pp->mc_runs + r0;                     // [k][e][r], e = LS, MMSE, MP, OMP
        if (rc == OFDM_OK) rc = ofdm_fft(ctx, Hmp, Hf, n, Nfft, 0);
        if (rc == OFDM_OK) rc = ofdm_interpolate(ctx, y, n, pc, Np, Nc, OFDM_INTERP_SPLINE, Hls);                     // LS_CE
        if (rc == OFDM_OK) rc = ofdm_mmse_ce_meas(ctx, y, n, pc, Np, Nc, hpad, Nc, snr_d, Hmm);
        if (rc == OFDM_OK) rc = ofdm_mp(ctx, y, n, Np, nullptr, pp->ldict_host[k], pc, Nfft, K, Hmp, nullptr, nullptr);
        if (rc == OFDM_OK)
            rc = ofdm_omp_ex(ctx, y, n, Np, nullptr, pp->ldict_host[k], pc, Nfft, K, Homp, nullptr, nullptr, nullptr, near, pp->tie_eps);
        if (rc == OFDM_OK) rc = ofdm_mse(ctx, Hf, Nfft, Hls, Nc, n, Nc, row);
        if (rc == OFDM_OK) rc = ofdm_mse(ctx, Hf, Nfft, Hmm, Nc, n, Nc, row + pp->mc_runs);
        if (rc == OFDM_OK) rc = ofdm_mse(ctx, Hf, Nfft, Hmp, Nfft, n, Nc, row + 2 * pp->mc_runs);
        if (rc == OFDM_OK) rc = ofdm_mse(ctx, Hf, Nfft, Homp, Nfft, n, Nc, row + 3 * pp->mc_runs);
        if (rc) return rc;
        int64_t* cnt = counts_dev + (size_t)k * 12;
        DISPATCH_T(ctx, {
            P2Est<T> est;
            est.H[0] = (const cx<T>*)Hls; est.H[1] = (const cx<T>*)Hmm; est.H[2] = (const cx<T>*)Hmp; est.H[3] = (const cx<T>*)Homp;
            est.stride[0] = Nc; est.stride[1] = Nc; est.stride[2] = Nfft; est.stride[3] = Nfft;
            part2_decide_kernel<T><<<dim3((unsigned)n, (unsigned)S), P2_THREADS, smem, ctx->stream>>>(
                (const cx<T>*)txn, L, (const cx<T>*)h, D, Nfft, ilog2(Nfft), Tg, (const cx<T>*)tw, dc0_dev, Nd, est,
                make_devconst<T>(base->constellation), pay_dev, stream_bits, (T)pp->near_eps, (unsigned long long*)cnt);
        });
        part2_runs_kernel<<<1, 256, 0, ctx->stream>>>(near, n, stream_bits, runs_dev + 2 * (size_t)k, cnt);
        ctx->launches += 2;
        return OFDM_OK;
    });
    return scr.finish(rc, "part-2 sweep launch failed");
}
