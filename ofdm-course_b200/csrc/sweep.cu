// ofdm_sweep_ber: the Monte-Carlo BER-vs-SNR sweep of the reference scripts as ONE library call per rank.
//
// Replaces the SNR loops `Task 3/Main_model_Task_3.m:192-268` and `Task 5/Main_model_Task_5.m:303-346` (chain 0:
// TX -> Noise -> multipath -> OFDM_demodulator -> LS_CE -> equalize -> demapping -> DeScrambler -> BER) and the
// impaired-channel chain of `Task 4/Main_model_Task_4.m:95-110,252-264,277-366` swept over SNR (chain 1:
// TX -> Noise -> add_STO -> add_CFO -> multipath -> AutoCorrFunction ... fine_sync -> estimate_channel -> BER).
//
// Work decomposition (SURVEY 8e): the global stream index g = snr_index * streams_per_point + j runs over
// n_snr * streams_per_point independent streams; rank r of `world` takes the contiguous share
// [T r / world, T (r+1) / world) -- equal to within one stream for ANY world size -- and walks it in tiles that never
// straddle an SNR point.  Payload bits, noise, STO and CFO draws are Philox streams keyed by g, so the integer
// counters do not depend on the number of ranks or on the tile size.  No data-path collective: the caller adds the
// counters of all ranks (one int64 all-reduce).  Everything is enqueued on the context's stream without any host
// synchronisation; the signal buffers are stream-ordered temporaries reused by every tile.
//
// The payload is drawn in the SCRAMBLED domain: the Philox words are the scrambled frames s, and the payload the chain is
// run on is p = DeScrambler(s) -- uniform because the scrambler is a bijection per frame, and Scrambler(p) = s exactly, so
// the TX chain on p with its scrambler IS the TX chain on s without it (checked bit for bit in
// tests/test_gpu_chain.py).  The three-tap descrambler runs at memory speed on 5 KB per stream, whereas the scrambler
// inside the TX kernel is eleven log-depth doublings per frame, a quarter of that kernel's time.
#include "philox.cuh"
#include "sweep_common.cuh"

uint32_t ofdm_reg_to_prev(const uint8_t* reg);

// payload words: word w of stream g = 32 Philox bits, counter (w/4, g), own key space
__global__ void payload_bits_kernel(uint32_t* __restrict__ bits, int64_t n_streams, int64_t words, uint64_t seed, int64_t first_stream) {
    const int64_t quads = (words + 3) >> 2;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_streams * quads) return;
    const int64_t b = i / quads, q = i - b * quads;
    const uint64_t g = (uint64_t)(first_stream + b);
    uint32_t c[4] = {(uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)g, (uint32_t)(g >> 32)};
    const uint64_t key = seed ^ 0x7061796c6f616421ULL;   // "payload!"
    philox4x32_10(c, (uint32_t)key, (uint32_t)(key >> 32));
    uint32_t* o = bits + b * words + 4 * q;
#pragma unroll
    for (int j = 0; j < 4; ++j) if (4 * q + j < words) o[j] = c[j];
}

// `Time_Delay = randi([0, Nfft + T_Guard])`, `Freq_Shift = randi([0, 30]) + (rand - 0.5)` (`Main_model_Task_4.m:101,108`)
__global__ void draw_sto_cfo_kernel(int64_t B, uint64_t seed, int64_t first_stream, int sto_max, int cfo_int_max, int32_t* __restrict__ nsto,
                                    double* __restrict__ cfo) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const uint64_t g = (uint64_t)(first_stream + b);
    uint32_t c[4] = {0u, 0u, (uint32_t)g, (uint32_t)(g >> 32)};
    const uint64_t key = seed ^ 0x73746f5f63666f21ULL;   // "sto_cfo!"
    philox4x32_10(c, (uint32_t)key, (uint32_t)(key >> 32));
    // multiply-shift maps a 32-bit word uniformly onto {0..m} (bias < 2^-21 for m <= 2048)
    if (nsto) nsto[b] = (int32_t)(((uint64_t)c[0] * (uint64_t)(sto_max + 1)) >> 32);
    if (cfo) cfo[b] = (double)(((uint64_t)c[1] * (uint64_t)(cfo_int_max + 1)) >> 32) + ((double)c[2] * 2.3283064365386963e-10 - 0.5);
}

// p = DeScrambler(s) for word-aligned streams, one thread per output word: out[i] = s[i] ^ s[i-13] ^ s[i-14] on a 64-bit
// window (previous word : this word); where a frame starts inside the window the bits below it are the initial register's
// history (`DeScrambler.m:8-13` with the per-frame reset of `Main_model_Task_4.m:350-364`).  Frames need not be word aligned.
__global__ void descramble_streams_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int64_t n_words, int words_per_stream,
                                          int frame_bits, uint32_t prev0) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    const int w = (int)(i % words_per_stream);                 // word inside its stream (streams are word aligned)
    const uint32_t R = in[i];
    out[i] = descramble_word(R, w ? in[i - 1] : 0u, w, frame_bits, prev0);
}

__global__ void fill_double_kernel(double* __restrict__ p, int64_t n, double v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

__global__ void sum_flags_kernel(const int32_t* __restrict__ f, int64_t n, unsigned long long* __restrict__ out) {
    int v = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) v += f[i] != 0;
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(out, (unsigned long long)v);
}

extern "C" int ofdm_payload_bits(ofdm_ctx* ctx, uint32_t* bits, int64_t n_streams, int64_t words_per_stream, uint64_t seed, int64_t first_stream_id) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, bits && n_streams >= 0 && words_per_stream > 0, "bad argument");
    if (n_streams == 0) return OFDM_OK;
    const int64_t n = n_streams * ((words_per_stream + 3) >> 2);
    payload_bits_kernel<<<(unsigned)cdiv64(n, 256), 256, 0, ctx->stream>>>(bits, n_streams, words_per_stream, seed, first_stream_id);
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_draw_sto_cfo(ofdm_ctx* ctx, int64_t B, uint64_t seed, int64_t first_stream_id, int sto_max, int cfo_int_max, int32_t* nsto_dev,
                                 double* cfo_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, B >= 0 && sto_max >= 0 && cfo_int_max >= 0 && (nsto_dev || cfo_dev), "bad argument");
    if (B == 0) return OFDM_OK;
    draw_sto_cfo_kernel<<<(unsigned)cdiv64(B, 256), 256, 0, ctx->stream>>>(B, seed, first_stream_id, sto_max, cfo_int_max, nsto_dev, cfo_dev);
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_sweep_share(int64_t total_streams, int rank, int world, int64_t* first, int64_t* count) {
    if (total_streams < 0 || world <= 0 || rank < 0 || rank >= world || !first || !count) return OFDM_ERR_INVALID;
    // 128-bit-safe for any realistic size: T < 2^40, world < 2^16
    const int64_t lo = total_streams * (int64_t)rank / world, hi = total_streams * (int64_t)(rank + 1) / world;
    *first = lo; *count = hi - lo;
    return OFDM_OK;
}

extern "C" int ofdm_sweep_ber(ofdm_ctx* ctx, const ofdm_link_params* lp, const ofdm_sweep_params* sp, int64_t* counts_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, lp && sp && counts_dev, "bad argument");
    REQUIRE(ctx, sp->n_snr > 0 && sp->snr_db_host && sp->streams_per_point > 0, "need at least one SNR point and one stream per point");
    REQUIRE(ctx, sp->world > 0 && sp->rank >= 0 && sp->rank < sp->world, "bad rank / world");
    REQUIRE(ctx, sp->chain == OFDM_SWEEP_TASK5 || sp->chain == OFDM_SWEEP_TASK4, "unknown chain");
    REQUIRE(ctx, sp->n_taps >= 0 && (sp->n_taps == 0 || sp->taps_host), "bad tap list");
    ConstTable ct = host_constellation(lp->constellation);
    REQUIRE(ctx, ct.bps > 0, "unknown constellation");
    const int64_t stream_bits = (int64_t)lp->S * lp->Nd * ct.bps;
    REQUIRE(ctx, stream_bits > 0 && stream_bits % 32 == 0, "the sweep needs word-aligned streams (S * Nd * bps divisible by 32)");
    REQUIRE(ctx, sp->chain == OFDM_SWEEP_TASK5 || ctx->precision == OFDM_PREC_F32, "the Task-4 sweep runs the fused FP32 chain");
    const int64_t words = stream_bits / 32;
    const int64_t L = (int64_t)lp->S * (lp->Nfft + lp->Tg);
    const size_t esz = ctx->precision == OFDM_PREC_F64 ? sizeof(double2) : sizeof(float2);

    // multipath impulse response on the device (`get_MP_channel_resp.m:2-19`), in the context's complex type
    void* h_dev = nullptr;
    int D = 0;
    if (sp->n_taps > 0) {
        std::vector<double> h;
        REQUIRE(ctx, sweep_dense_taps(sp->taps_host, sp->n_taps, 4096, h), "tap delays must be integers in [0, 4096)");
        D = (int)h.size();
        std::vector<double> hd(2 * (size_t)D, 0.0);
        for (int d = 0; d < D; ++d) hd[2 * (size_t)d] = h[d];
        if (ctx->precision == OFDM_PREC_F64) h_dev = ctx_blob(ctx, hd.data(), sizeof(double) * hd.size());
        else { std::vector<float> hf(hd.begin(), hd.end()); h_dev = ctx_blob(ctx, hf.data(), sizeof(float) * hf.size()); }
        REQUIRE(ctx, h_dev != nullptr, "device upload failed");
    }

    const void* unit_tap = nullptr;                                           // "no multipath" for the fused Task-4 channel
    if (sp->chain == OFDM_SWEEP_TASK4 && !h_dev) {
        const double one_d[2] = {1.0, 0.0};
        const float one_f[2] = {1.f, 0.f};
        unit_tap = ctx->precision == OFDM_PREC_F64 ? ctx_blob(ctx, one_d, sizeof one_d) : ctx_blob(ctx, one_f, sizeof one_f);
        REQUIRE(ctx, unit_tap != nullptr, "device upload failed");
    }
    // whole tiles of 8,192 streams keep the persistent kernels' tails below 1 %
    const SweepTiles tiles(sp->n_snr, sp->streams_per_point, sp->rank, sp->world, sp->tile_streams, 8192);
    if (tiles.count == 0) return OFDM_OK;
    const int64_t tile = tiles.tile;

    // stream-ordered temporaries, sized for one tile and reused by every tile of the call
    const bool t4 = sp->chain == OFDM_SWEEP_TASK4;
    const size_t sig_b = esz * (size_t)L * tile, bits_b = sizeof(uint32_t) * (size_t)words * tile, d_b = sizeof(double) * tile, i_b = sizeof(int32_t) * tile;
    SweepScratch scr(ctx);
    CUDA_TRY(ctx, scr.alloc({sig_b, sig_b, t4 ? sig_b : 0, bits_b, bits_b, d_b, d_b, d_b, i_b, i_b}));
    void* tx = scr.get<void>(0);
    void* rx = scr.get<void>(1);
    void* tmp = t4 ? scr.get<void>(2) : nullptr;
    uint32_t* sbits = scr.get<uint32_t>(3);                                 // scrambled frames s (Philox)
    uint32_t* bits = lp->scramble ? scr.get<uint32_t>(4) : sbits;           // payload p = DeScrambler(s): the reference bits (no scrambler: p = s)
    double* snr_d = scr.get<double>(5);
    double* psum = scr.get<double>(6);
    double* cfo_d = scr.get<double>(7);
    int32_t* sto_d = scr.get<int32_t>(8);
    int32_t* fail_d = scr.get<int32_t>(9);
    ofdm_link_params lp_tx = *lp;                                           // the TX side maps s directly
    lp_tx.scramble = 0;

    const int rc = tiles.walk([&](int64_t i, int64_t, int64_t g, int64_t n) {   // i: SNR point of this tile
        int64_t* row = counts_dev + 4 * i;
        int rc = ofdm_sweep_tile_payload(ctx, lp, sbits, bits, n, words, sp->seed, g);
        if (rc) return rc;
        fill_double_kernel<<<(unsigned)cdiv64(n, 256), 256, 0, ctx->stream>>>(snr_d, n, sp->snr_db_host[i]);
        ctx->launches++;
        if (!t4) {
            // Task 5 order: Noise, then multipath (`Main_model_Task_5.m:108,123-127`)
            rc = ofdm_tx_chain_p(ctx, &lp_tx, sbits, n, tx, psum);
            if (rc == OFDM_OK) rc = ofdm_channel_t5_p(ctx, tx, n, L, snr_d, psum, nullptr, sp->seed, g, h_dev, D, rx);
            if (rc == OFDM_OK) rc = ofdm_rx_chain_t5(ctx, lp, rx, n, bits, nullptr, nullptr, row, nullptr, sp->near_eps);
        } else {
            // Task 4 order: Noise -> add_STO -> add_CFO -> multipath (`Main_model_Task_4.m:95,103,110,263-264`)
            const void* rxs = tx;                                           // where the received streams end up
            rc = ofdm_tx_chain_p(ctx, &lp_tx, sbits, n, tx, psum);
            if (rc == OFDM_OK) rc = ofdm_draw_sto_cfo(ctx, n, sp->seed, g, sp->sto_max, sp->cfo_int_max, sto_d, cfo_d);
            if (rc == OFDM_OK && D <= 1024 && !getenv("OFDM_B200_T4_CHANNEL_COMPOSED")) {
                // one pass: the four impairments fused (bit-identical to the composition below)
                rc = ofdm_channel_t4_p(ctx, tx, n, L, snr_d, psum, nullptr, sp->seed, g, sto_d, cfo_d, lp->Nfft, h_dev ? h_dev : unit_tap, h_dev ? D : 1, rx);
                rxs = rx;
            } else {
                if (rc == OFDM_OK) rc = ofdm_add_noise(ctx, tx, n, L, snr_d, nullptr, sp->seed, g, rx, nullptr);
                if (rc == OFDM_OK) rc = ofdm_add_sto(ctx, rx, n, L, sto_d, tmp);
                if (rc == OFDM_OK) rc = ofdm_add_cfo(ctx, tmp, n, L, cfo_d, lp->Nfft, h_dev ? rx : tx);
                if (rc == OFDM_OK && h_dev) rc = ofdm_apply_fir(ctx, rx, n, L, h_dev, D, 0, tx);
            }
            if (rc == OFDM_OK) rc = ofdm_rx_chain_t4_ex(ctx, lp, rxs, n, 1, 1, h_dev ? 1 : 0, bits, nullptr, row, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                                        sp->near_eps, fail_d);
            if (rc == OFDM_OK) {
                sum_flags_kernel<<<(unsigned)std::min<int64_t>(cdiv64(n, 256), 64), 256, 0, ctx->stream>>>(fail_d, n, (unsigned long long*)(row + 3));
                ctx->launches++;
            }
        }
        return rc;
    });
    return scr.finish(rc, "sweep launch failed");
}

// The payload of streams g .. g + n - 1 exactly as ofdm_sweep_ber draws it (not exported): Philox words s into sbits, and
// p = DeScrambler(s) into bits when the chain scrambles (otherwise p = s and bits is not written).
int ofdm_sweep_tile_payload(ofdm_ctx* ctx, const ofdm_link_params* lp, uint32_t* sbits, uint32_t* bits, int64_t n, int64_t words, uint64_t seed, int64_t g) {
    int rc = ofdm_payload_bits(ctx, sbits, n, words, seed, g);
    if (rc != OFDM_OK || !lp->scramble) return rc;
    const int64_t frames = lp->S / lp->SpF, frame_bits = 32 * words / frames;
    if (frame_bits >= 64) {
        descramble_streams_kernel<<<(unsigned)cdiv64(n * words, 256), 256, 0, ctx->stream>>>(sbits, bits, n * words, (int)words, (int)frame_bits,
                                                                                             ofdm_reg_to_prev(lp->reg0_host));
        ctx->launches++;
        return OFDM_OK;
    }
    return ofdm_descramble(ctx, sbits, bits, n * frames, frame_bits, lp->reg0_host, nullptr);
}
