// ofdm_sweep_papr: the Task-2 PAPR study (`Task 2/Main_model_Task_2.m:72-82`) as ONE library call per rank.
//
// Task 2 compares the PAPR of the transmitted signal with and without the scrambler: the PAPR of the whole serial stream
// (calculatePAPR, `Task 2/README.md:54`) and the CCDF of the PAPR of every Nfft-sample window (calculate_window_PAPR ->
// calculateCCDF, `README.md:69-71`).  Work item g = k * streams_per_point + j over points k (a scramble flag and a payload
// source) and streams j; the rank's share (ofdm_sweep_share) is walked in tiles that never straddle a point, as the other
// sweeps do.  Per tile: the payload (Bernoulli bits from Philox, or a window of a caller's pool), ofdm_tx_chain_p with the
// point's scramble flag, then papr_stats_kernel (papr.cu), which turns the TX streams into the point's window-PAPR histogram
// and the per-stream PAPR without storing a window value.  The payload depends on j only, so the points of one study
// transmit the same payloads: plain against scrambled is a paired comparison, as the reference's one image is.
#include "philox.cuh"
#include "sweep_common.cuh"

#include <cmath>

int ofdm_papr_stats_check(ofdm_ctx* ctx, int W, int n_bins, const char* who);
int ofdm_papr_stats(ofdm_ctx* ctx, const void* x, int64_t B, int64_t L, int W, const double* psum, double bin_db, int n_bins, int64_t* hist,
                    double* papr, unsigned long long* peak);

// Bernoulli payload written straight into one contiguous bitstream (streams need not be word aligned), one thread per word:
// bit i of stream s is 1 iff u_i < thr, u_i = word i mod 4 of Philox4x32-10 at counter (i / 4, first + s) in its own key space.
// Bits past the last stream are 0.
__global__ void bernoulli_bits_kernel(uint32_t* __restrict__ out, int64_t total_bits, int64_t stream_bits, uint32_t thr, uint64_t seed, int64_t first) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (32 * w >= total_bits) return;
    const uint64_t key = seed ^ 0x6265726e6f756c6cULL;   // "bernoull"
    int64_t s = (32 * w) / stream_bits, i = 32 * w - s * stream_bits;
    int64_t q_have = -1, s_have = -1;
    uint32_t c[4] = {0u, 0u, 0u, 0u};
    uint32_t v = 0;
    for (int t = 0; t < 32 && 32 * w + t < total_bits; ++t, ++i) {
        if (i == stream_bits) { ++s; i = 0; }
        const int64_t q = i >> 2;
        if (q != q_have || s != s_have) {
            const uint64_t g = (uint64_t)(first + s);
            c[0] = (uint32_t)q; c[1] = (uint32_t)((uint64_t)q >> 32); c[2] = (uint32_t)g; c[3] = (uint32_t)(g >> 32);
            philox4x32_10(c, (uint32_t)key, (uint32_t)(key >> 32));
            q_have = q; s_have = s;
        }
        const int r = (int)(i & 3);
        if ((r == 0 ? c[0] : r == 1 ? c[1] : r == 2 ? c[2] : c[3]) < thr) v |= 1u << t;   // (no local-memory array)
    }
    out[w] = v;
}

// Pool payload into one contiguous bitstream: bit i of stream s is pool bit (((first + s) * stride + i) mod pool_bits),
// copied a run of consecutive pool bits at a time.  Bits past the last stream are 0.  pool_bits <= 2^32, stride < pool_bits.
__global__ void pool_bits_kernel(const uint32_t* __restrict__ pool, int64_t pool_bits, int64_t stride, uint32_t* __restrict__ out, int64_t total_bits,
                                 int64_t stream_bits, int64_t first) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (32 * w >= total_bits) return;
    const uint64_t pb = (uint64_t)pool_bits;
    uint32_t v = 0;
    for (int t = 0; t < 32 && 32 * w + t < total_bits;) {
        const int64_t P = 32 * w + t, s = P / stream_bits, i = P - s * stream_bits;
        const int64_t src = (int64_t)(((uint64_t)(first + s) % pb * (uint64_t)stride + (uint64_t)i % pb) % pb);
        const int take = (int)min(min((int64_t)(32 - t), stream_bits - i), min(pool_bits - src, total_bits - P));
        uint32_t u = bits_get32(pool, src, pool_bits);
        if (take < 32) u &= (1u << take) - 1u;
        v |= u << t;
        t += take;
    }
    out[w] = v;
}

static int bernoulli_launch(ofdm_ctx* ctx, uint32_t* bits, int64_t n_streams, int64_t stream_bits, double p_one, uint64_t seed, int64_t first) {
    const int64_t total = n_streams * stream_bits;
    const uint32_t thr = (uint32_t)floor(p_one * 4294967296.0);
    bernoulli_bits_kernel<<<(unsigned)cdiv64(cdiv64(total, 32), 256), 256, 0, ctx->stream>>>(bits, total, stream_bits, thr, seed, first);
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

extern "C" int ofdm_payload_bernoulli(ofdm_ctx* ctx, uint32_t* bits_dev, int64_t n_streams, int64_t stream_bits, double p_one, uint64_t seed,
                                      int64_t first_stream_id) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, bits_dev, "bits_dev is NULL");
    REQUIRE(ctx, n_streams >= 0, "n_streams must be >= 0");
    REQUIRE(ctx, stream_bits >= 1, "stream_bits must be >= 1");
    REQUIRE(ctx, p_one > 0.0 && p_one < 1.0, "p_one must lie in (0, 1)");
    REQUIRE(ctx, first_stream_id >= 0, "first_stream_id must be >= 0");
    if (n_streams == 0) return OFDM_OK;
    return bernoulli_launch(ctx, bits_dev, n_streams, stream_bits, p_one, seed, first_stream_id);
}

extern "C" int ofdm_sweep_papr(ofdm_ctx* ctx, const ofdm_link_params* lp, const ofdm_papr_params* pp, double* papr_dev, int64_t* hist_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, lp, "ofdm_sweep_papr: link parameters are NULL");
    REQUIRE(ctx, pp, "ofdm_sweep_papr: PAPR parameters are NULL");
    REQUIRE(ctx, papr_dev, "ofdm_sweep_papr: papr_dev is NULL");
    REQUIRE(ctx, hist_dev, "ofdm_sweep_papr: hist_dev is NULL");
    REQUIRE(ctx, pp->n_points > 0, "ofdm_sweep_papr: need at least one point");
    REQUIRE(ctx, pp->scramble_host, "ofdm_sweep_papr: scramble_host is NULL");
    for (int k = 0; k < pp->n_points; ++k) REQUIRE(ctx, pp->scramble_host[k] == 0 || pp->scramble_host[k] == 1, "ofdm_sweep_papr: scramble flags must be 0 or 1");
    if (pp->pool_host) {
        REQUIRE(ctx, pp->pool_bits >= 1 && pp->pool_bits <= ((int64_t)1 << 32), "ofdm_sweep_papr: pool_bits must lie in 1..2^32");
        REQUIRE(ctx, pp->pool_stride >= 0, "ofdm_sweep_papr: pool_stride must be >= 0");
    } else {
        REQUIRE(ctx, pp->p_one_host, "ofdm_sweep_papr: p_one_host is NULL (and no pool)");
        for (int k = 0; k < pp->n_points; ++k) REQUIRE(ctx, pp->p_one_host[k] > 0.0 && pp->p_one_host[k] < 1.0, "ofdm_sweep_papr: p_one must lie in (0, 1)");
    }
    REQUIRE(ctx, pp->streams_per_point > 0, "ofdm_sweep_papr: need at least one stream per point");
    REQUIRE(ctx, pp->tile_streams >= 0, "ofdm_sweep_papr: tile_streams must be >= 0 (0 = default)");
    REQUIRE(ctx, pp->world > 0 && pp->rank >= 0 && pp->rank < pp->world, "ofdm_sweep_papr: rank must lie in 0..world-1");
    REQUIRE(ctx, pp->bin_db > 0.0 && std::isfinite(pp->bin_db), "ofdm_sweep_papr: bin_db must be a finite width > 0");
    REQUIRE(ctx, pp->n_bins >= 1 && pp->n_bins <= 16384, "ofdm_sweep_papr: n_bins must lie in 1..16384");
    ConstTable ct = host_constellation(lp->constellation);
    REQUIRE(ctx, ct.bps > 0, "ofdm_sweep_papr: unknown constellation");
    REQUIRE(ctx, lp->S > 0 && lp->SpF > 0 && lp->S % lp->SpF == 0, "ofdm_sweep_papr: S must be a positive multiple of SpF");
    REQUIRE(ctx, is_pow2(lp->Nfft) && lp->Nfft >= 8 && lp->Nfft <= (ctx->precision == OFDM_PREC_F64 ? 4096 : 8192),
            "ofdm_sweep_papr: Nfft must be a power of two the TX chain takes (8..8192 in FP32, 8..4096 in FP64)");
    REQUIRE(ctx, lp->Tg >= 0 && lp->Tg <= lp->Nfft, "ofdm_sweep_papr: T_Guard must lie in 0..Nfft");
    REQUIRE(ctx, lp->Nd >= 1, "ofdm_sweep_papr: need at least one data carrier");
    int rc = ofdm_papr_stats_check(ctx, lp->Nfft, pp->n_bins, "ofdm_sweep_papr");
    if (rc) return rc;
    const int64_t stream_bits = (int64_t)lp->S * lp->Nd * ct.bps;
    const int64_t L = (int64_t)lp->S * (lp->Nfft + lp->Tg);
    const int64_t spp = pp->streams_per_point;

    const SweepTiles tiles(pp->n_points, spp, pp->rank, pp->world, pp->tile_streams, 8192);   // 3.8 GB of FP32 signal at the Task-2 shape
    if (tiles.count == 0) return OFDM_OK;
    const int64_t tile = tiles.tile;

    // one stream-ordered allocation per call: signal, payload, power sums, maxima and (when given) the pool.  The pool is
    // not put in the context's blob cache: a call must not evict other tables, nor keep a large pool alive after it returns.
    const size_t esz = ctx->precision == OFDM_PREC_F64 ? sizeof(double2) : sizeof(float2);
    const int64_t pool_words = pp->pool_host ? cdiv64(pp->pool_bits, 32) : 0;
    SweepScratch scr(ctx);
    CUDA_TRY(ctx, scr.alloc({esz * (size_t)L * tile, sizeof(uint32_t) * (size_t)(cdiv64(tile * stream_bits, 32) + 1), sizeof(double) * tile,
                             sizeof(double) * tile, sizeof(uint32_t) * (size_t)pool_words}));
    void* tx = scr.get<void>(0);
    uint32_t* bits = scr.get<uint32_t>(1);
    double* psum = scr.get<double>(2);
    unsigned long long* peak = scr.get<unsigned long long>(3);
    uint32_t* pool = pp->pool_host ? scr.get<uint32_t>(4) : nullptr;
    if (pool) rc = cudaMemcpyAsync(pool, pp->pool_host, sizeof(uint32_t) * (size_t)pool_words, cudaMemcpyHostToDevice, ctx->stream) == cudaSuccess
                       ? OFDM_OK : ctx_fail(ctx, OFDM_ERR_CUDA, "ofdm_sweep_papr: pool upload failed");
    const int64_t stride = pp->pool_host ? pp->pool_stride % pp->pool_bits : 0;

    ofdm_link_params lpk = *lp;
    if (rc == OFDM_OK) rc = tiles.walk([&](int64_t k, int64_t j0, int64_t g, int64_t n) {   // point and first stream of this tile
        int rc = OFDM_OK;
        if (pool) {
            const int64_t total = n * stream_bits;
            pool_bits_kernel<<<(unsigned)cdiv64(cdiv64(total, 32), 256), 256, 0, ctx->stream>>>(pool, pp->pool_bits, stride, bits, total, stream_bits, j0);
            ctx->launches++;
        } else rc = bernoulli_launch(ctx, bits, n, stream_bits, pp->p_one_host[k], pp->seed, j0);
        lpk.scramble = pp->scramble_host[k];
        if (rc == OFDM_OK) rc = ofdm_tx_chain_p(ctx, &lpk, bits, n, tx, psum);
        if (rc == OFDM_OK)
            rc = ofdm_papr_stats(ctx, tx, n, L, lp->Nfft, psum, pp->bin_db, pp->n_bins, hist_dev + k * pp->n_bins, papr_dev + g, peak);
        return rc;
    });
    return scr.finish(rc, "ofdm_sweep_papr launch failed");
}
