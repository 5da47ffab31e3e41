// ofdm_sweep_sync: the Task-4 synchroniser and channel-estimate accuracy study over SNR as ONE library call per rank.
//
// Task 4 (`Task 4/Main_model_Task_4.m:95-110,277-374`) reports, besides BER, how well AutoCorrFunction finds the symbol start
// and the CFO (`Task 4/README.md:111-121`), the NMSE of the pilot-step-4 channel estimate over SNR (`Task 4/graphs/nmse(snr).png`)
// and the MER of every run (`:374`).  This call runs the Task-4 chain of ofdm_sweep_ber -- same share rule (ofdm_sweep_share),
// stream numbering g = snr_index * streams_per_point + j, tiles that never straddle a point, and the Philox keys of the
// payload, noise and STO / CFO draws -- so with sto_mode 0 and every desync flag on it transmits the same streams.  The
// receiver is the split Task-4 chain with the statistics variant of its last kernel (chain_rx_t4.cu: t4_post_kernel's STATS),
// which writes one record per stream and adds to the point's counters; the estimated response is never stored.
// Streams need not be word aligned (Task 4 at 25 % pilots: 59,800 bits): stream g then carries the first stream_bits bits of
// the Philox words ofdm_payload_bits draws for it (ceil(stream_bits / 32) words), packed into one contiguous bitstream.
// Every record cell is written by exactly one rank, counters are integer atomics, so the caller's sums over ranks are exact.
#include "sweep_common.cuh"

int ofdm_rx_t4_sync_stats(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx, int64_t B, int time_desync, int freq_desync, int mp_desync,
                          const uint32_t* tx_bits, int64_t* row, int32_t* tg, double* fo, int32_t* ifo, int32_t* fail, const int32_t* nsto,
                          const double* cfo, const double* Htrue_dev, double* rec, int64_t rec_stride);

// per stream of a tile: the SNR the channel reads and, with fixed impairments (sto_mode 1), the STO and CFO
__global__ void sync_fill_kernel(int64_t n, double snr_db, double* __restrict__ snr, int fixed, int32_t sto, double cfo, int32_t* __restrict__ nsto,
                                 double* __restrict__ cfo_out) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    snr[b] = snr_db;
    if (fixed) { nsto[b] = sto; cfo_out[b] = cfo; }
}

// contiguous bitstream of n streams of stream_bits bits from per-stream padded words (wpad words per stream)
__global__ void sync_pack_kernel(const uint32_t* __restrict__ in, int64_t wpad, int64_t stream_bits, int64_t total_bits, uint32_t* __restrict__ out) {
    const int64_t W = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (32 * W >= total_bits) return;
    uint32_t v = 0;
    for (int t = 0; t < 32;) {
        const int64_t i = 32 * W + t;
        if (i >= total_bits) break;
        const int64_t b = i / stream_bits, o = i - b * stream_bits;
        const int take = (int)min(min((int64_t)(32 - t), stream_bits - o), (int64_t)(32 - (o & 31)));   // bits left in this input word
        uint32_t wv = in[b * wpad + (o >> 5)] >> (o & 31);
        if (take < 32) wv &= (1u << take) - 1u;
        v |= wv << t;
        t += take;
    }
    out[W] = v;
}

void ofdm_sweep_fill(ofdm_ctx* ctx, int64_t n, double snr_db, int fixed, int32_t sto, double cfo, double* snr, int32_t* nsto, double* cfo_out) {
    sync_fill_kernel<<<(unsigned)cdiv64(n, 256), 256, 0, ctx->stream>>>(n, snr_db, snr, fixed, sto, cfo, nsto, cfo_out);
    ctx->launches++;
}

void ofdm_sweep_pack_bits(ofdm_ctx* ctx, const uint32_t* raw, int64_t n, int64_t wpad, int64_t stream_bits, uint32_t* out) {
    sync_pack_kernel<<<(unsigned)cdiv64(n * wpad, 256), 256, 0, ctx->stream>>>(raw, wpad, stream_bits, n * stream_bits, out);
    ctx->launches++;
}

extern "C" int ofdm_sweep_sync(ofdm_ctx* ctx, const ofdm_link_params* lp, const ofdm_sync_params* sp, double* rec_dev, int64_t* counts_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, lp, "ofdm_sweep_sync: link parameters are NULL");
    REQUIRE(ctx, sp, "ofdm_sweep_sync: sync parameters are NULL");
    REQUIRE(ctx, rec_dev, "ofdm_sweep_sync: rec_dev is NULL");
    REQUIRE(ctx, counts_dev, "ofdm_sweep_sync: counts_dev is NULL");
    if (ctx->precision != OFDM_PREC_F32) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "ofdm_sweep_sync runs the FP32 Task-4 chain only (context is FP64)");
    if (lp->Nfft != 1024) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "ofdm_sweep_sync supports Nfft = 1024 only (got %d)", lp->Nfft);
    REQUIRE(ctx, sp->n_snr > 0, "ofdm_sweep_sync: need at least one SNR point");
    REQUIRE(ctx, sp->snr_db_host, "ofdm_sweep_sync: snr_db_host is NULL");
    REQUIRE(ctx, sp->streams_per_point > 0, "ofdm_sweep_sync: need at least one stream per point");
    REQUIRE(ctx, sp->tile_streams >= 0, "ofdm_sweep_sync: tile_streams must be >= 0 (0 = default)");
    REQUIRE(ctx, sp->world > 0 && sp->rank >= 0 && sp->rank < sp->world, "ofdm_sweep_sync: rank must lie in 0..world-1");
    REQUIRE(ctx, sp->n_taps >= 0 && (sp->n_taps == 0 || sp->taps_host), "ofdm_sweep_sync: bad tap list");
    REQUIRE(ctx, sp->sto_mode == 0 || sp->sto_mode == 1, "ofdm_sweep_sync: sto_mode must be 0 (drawn) or 1 (fixed)");
    REQUIRE(ctx, sp->sto_mode == 1 || (sp->sto_max >= 0 && sp->cfo_int_max >= 0), "ofdm_sweep_sync: sto_max and cfo_int_max must be >= 0");
    REQUIRE(ctx, sp->sto_mode == 0 || (sp->sto_fixed >= 0 && std::isfinite(sp->cfo_fixed)), "ofdm_sweep_sync: sto_fixed must be >= 0 and cfo_fixed finite");
    ConstTable ct = host_constellation(lp->constellation);
    REQUIRE(ctx, ct.bps > 0, "ofdm_sweep_sync: unknown constellation");
    REQUIRE(ctx, lp->S > 0 && lp->SpF > 0 && lp->S % lp->SpF == 0, "ofdm_sweep_sync: S must be a positive multiple of SpF");
    REQUIRE(ctx, lp->N_carrier >= 2 && lp->N_carrier <= lp->Nfft, "ofdm_sweep_sync: N_carrier must lie in 2..Nfft");
    REQUIRE(ctx, lp->Tg >= 0 && lp->Tg <= lp->Nfft, "ofdm_sweep_sync: T_Guard must lie in 0..Nfft");
    REQUIRE(ctx, lp->Np >= 2 && lp->Nd >= 1, "ofdm_sweep_sync: need at least two pilots and one data carrier");
    const int64_t stream_bits = (int64_t)lp->S * lp->Nd * ct.bps;
    const bool aligned = stream_bits % 32 == 0;
    const int Nfft = lp->Nfft, Nc = lp->N_carrier;
    const int64_t words = (stream_bits + 31) / 32;                                  // Philox words per stream
    const int64_t L = (int64_t)lp->S * (Nfft + lp->Tg);

    // the channel: impulse response in FP32 for the channel kernel, and the true response H(1:N_carrier) in double
    // (`get_MP_channel_resp.m:2-19`: later rows overwrite; H = fft(h, Nfft)), one table per call
    std::vector<double> h(1, 1.0);                                                  // no multipath: a single unit tap, H = 1
    if (sp->n_taps > 0)
        REQUIRE(ctx, sweep_dense_taps(sp->taps_host, sp->n_taps, Nfft, h), "ofdm_sweep_sync: tap delays must be integers in [0, Nfft)");
    const int D = (int)h.size();
    std::vector<float> hf(2 * (size_t)D, 0.f);
    for (int d = 0; d < D; ++d) hf[2 * d] = (float)h[d];
    std::vector<double> Ht(2 * (size_t)Nc, 0.0);
    for (int k = 0; k < Nc; ++k) {
        double re = 0.0, im = 0.0;
        for (int d = 0; d < D; ++d) {
            if (h[d] == 0.0) continue;
            const double a = -2.0 * M_PI * (double)(((int64_t)d * k) % Nfft) / Nfft;
            re += h[d] * cos(a);
            im += h[d] * sin(a);
        }
        Ht[2 * k] = re; Ht[2 * k + 1] = im;
    }
    const void* h_dev = ctx_blob(ctx, hf.data(), sizeof(float) * hf.size());
    const double* Ht_dev = (const double*)ctx_blob(ctx, Ht.data(), sizeof(double) * Ht.size());
    REQUIRE(ctx, h_dev && Ht_dev, "ofdm_sweep_sync: device upload failed");

    SweepTiles tiles(sp->n_snr, sp->streams_per_point, sp->rank, sp->world, sp->tile_streams, 8192);
    if (tiles.count == 0) return OFDM_OK;
    if (!aligned) tiles.tile = std::min<int64_t>(tiles.tile, 16384);               // the receiver takes unaligned streams in one pass
    const int64_t tile = tiles.tile;

    // stream-ordered temporaries, sized for one tile and reused by every tile of the call
    const size_t b_sig = sizeof(float2) * (size_t)L * tile, b_bits = sizeof(uint32_t) * (size_t)(words + 1) * tile, b_d = sizeof(double) * tile,
                 b_i = sizeof(int32_t) * tile;
    SweepScratch scr(ctx);
    CUDA_TRY(ctx, scr.alloc({b_sig, b_sig, b_bits, b_bits, b_d, b_d, b_d, b_d, b_i, b_i, b_i, b_i, aligned ? 0 : b_bits}));
    void* tx = scr.get<void>(0);
    void* rx = scr.get<void>(1);
    uint32_t* sbits = scr.get<uint32_t>(2);                                          // scrambled frames s (Philox)
    uint32_t* bits = lp->scramble ? scr.get<uint32_t>(3) : sbits;                    // payload p = DeScrambler(s)
    double* snr_d = scr.get<double>(4);
    double* psum = scr.get<double>(5);
    double* cfo_d = scr.get<double>(6);
    double* fo_d = scr.get<double>(7);
    int32_t* sto_d = scr.get<int32_t>(8);
    int32_t* tg_d = scr.get<int32_t>(9);
    int32_t* ifo_d = scr.get<int32_t>(10);
    int32_t* fail_d = scr.get<int32_t>(11);
    uint32_t* raw = scr.get<uint32_t>(12);                                           // padded Philox words of unaligned streams
    ofdm_link_params lp_tx = *lp;                                                    // as ofdm_sweep_ber: the TX maps s directly
    lp_tx.scramble = 0;

    const int64_t spp = sp->streams_per_point;
    const int rc = tiles.walk([&](int64_t i, int64_t j0, int64_t g, int64_t n) {      // i: SNR point of this tile
        int rc;
        if (aligned) rc = ofdm_sweep_tile_payload(ctx, lp, sbits, bits, n, words, sp->seed, g);
        else {
            rc = ofdm_payload_bits(ctx, raw, n, words, sp->seed, g);
            if (rc == OFDM_OK) ofdm_sweep_pack_bits(ctx, raw, n, words, stream_bits, sbits);
            if (rc == OFDM_OK && lp->scramble) rc = ofdm_descramble(ctx, sbits, bits, n * (lp->S / lp->SpF), stream_bits / (lp->S / lp->SpF), lp->reg0_host, nullptr);
        }
        if (rc) return rc;
        ofdm_sweep_fill(ctx, n, sp->snr_db_host[i], sp->sto_mode, sp->sto_fixed, sp->cfo_fixed, snr_d, sto_d, cfo_d);
        // Task 4 order: Noise -> add_STO -> add_CFO -> multipath (`Main_model_Task_4.m:95,103,110,263-264`), one pass
        rc = ofdm_tx_chain_p(ctx, &lp_tx, sbits, n, tx, psum);
        if (rc == OFDM_OK && sp->sto_mode == 0) rc = ofdm_draw_sto_cfo(ctx, n, sp->seed, g, sp->sto_max, sp->cfo_int_max, sto_d, cfo_d);
        if (rc == OFDM_OK) rc = ofdm_channel_t4_p(ctx, tx, n, L, snr_d, psum, nullptr, sp->seed, g, sto_d, cfo_d, Nfft, h_dev, D, rx);
        if (rc == OFDM_OK)
            rc = ofdm_rx_t4_sync_stats(ctx, lp, rx, n, sp->time_desync, sp->freq_desync, sp->mp_desync, bits, counts_dev + 4 * i, tg_d, fo_d, ifo_d, fail_d,
                                       sto_d, cfo_d, Ht_dev, rec_dev + i * 9 * spp + j0, spp);
        return rc;
    });
    return scr.finish(rc, "ofdm_sweep_sync launch failed");
}
