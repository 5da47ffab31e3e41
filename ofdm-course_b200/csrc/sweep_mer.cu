// ofdm_sweep_mer: the Task-3 BER and MER study over constellations and SNR as ONE library call per rank.
//
// Task 3 (`Task 3/Main_model_Task_3.m:192-268`, `Task 3/README.md:53-55`) draws the BER-vs-SNR curves of BPSK, QPSK, 8PSK and
// 16QAM and prints the MER, with a receiver that has no synchroniser, estimator or equaliser: OFDM_demodulator ->
// get_payload -> demapping -> DeScrambler -> BER_func, and MER_func on the same data carriers.  Each point of the call has
// its own constellation, SNR and fixed STO / CFO; stream numbering, tiles, payload and channel keys are those of
// ofdm_sweep_sync (sweep_sync.cu), so with one constellation, equal pilots and sto_mode 1 both calls transmit the same streams.
//
// The receiver, rx_t3_kernel, decides every symbol in the pass that transforms it; nothing is written per symbol:
//   * one CTA per stream, one warp per OFDM symbol (warp w takes symbols w, w + 8, ...): the 1024 samples after the cyclic
//     prefix (the prefix is never read), the split Task-4 chain's 1024-point transform (t4_load_window / t4_pass_a / fft32
//     of rx1024.cuh, as t4_sym_kernel runs it with every desync flag off), so bins and decisions are bit-identical to
//     those of ofdm_rx_chain_t4_ex(..., 0, 0, 0, ...) when that call takes its split chain (from 512 streams on, for shapes
//     whose fused kernel fits in 111 KB of shared memory; its fused and generic kernels round differently);
//   * the data carriers of the symbol are decided by its warp (16QAM: the separable rule of demap16_nib; BPSK / QPSK / 8PSK:
//     the first-minimum table rule of nearest_idx), with the near-boundary count of ofdm_demap and the two MER_func sums
//     `MER_func.m:7-25` in double;
//   * bit errors without a descrambled copy: the CTA holds e = d XOR s, the decided bits d XORed into the stream's
//     transmitted scrambled bits s, in shared memory, and counts popcount(e[i] ^ e[i-13] ^ e[i-14]) with zero history at
//     every frame start.  DeScrambler is affine and both DeScrambler(d) and the payload p = DeScrambler(s) start from the same
//     register, so the register terms cancel and this is the error count of DeScrambler(d) against p.
// Every MER sum is accumulated per thread in symbol order and reduced with the fixed-order block_sum: its value depends on
// the stream shape only, never on the tile, rank or world.
#include "rx1024.cuh"
#include "sweep_common.cuh"

#define T3_THREADS 256

struct T3Params {
    int Tg, Nc, S, Nd, bps, frame_bits, frames, scramble;
    const int32_t* data0;      // Nd 0-based data carriers
};

// The shared-memory error words of one stream: d XOR s, bit i of the stream at word i / 32, bit i % 32.
__device__ __forceinline__ void t3_xor_bits(uint32_t* ew, int64_t pos, int n, uint32_t bits) {
    const int sh = (int)(pos & 31);
    atomicXor(&ew[pos >> 5], bits << sh);
    if (sh + n > 32) atomicXor(&ew[(pos >> 5) + 1], bits >> (32 - sh));
}

// One CTA per stream of B.  s: the stream's scrambled words, wpad per stream (the first stream_bits bits are the stream);
// mer: f0 at mer[b], f1 at mer[mer_stride + b]; counts {errors, bits, near-boundary symbols} +=.
template <int K2N, bool QAM16>
__global__ void __launch_bounds__(T3_THREADS, 2) rx_t3_kernel(T3Params p, T4FastExtra fx, DevConst<float> con, float a_in, float a_out,
                                                              const float2* __restrict__ rx, int64_t L, const uint32_t* __restrict__ s,
                                                              int64_t wpad, double* __restrict__ mer, int64_t mer_stride,
                                                              unsigned long long* __restrict__ counts, float near_eps) {
    constexpr int N = 1024, NW = T3_THREADS / 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double red[32];
    __shared__ int red_i[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b = blockIdx.x;
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
    const int words = (int)((stream_bits + 31) >> 5);
    __shared__ int near_s;
    float2* E = (float2*)smem_raw + warp * 32 * T4F_EROW;
    uint32_t* ew = (uint32_t*)((float2*)smem_raw + NW * 32 * T4F_EROW);
    for (int w = tid; w < words; w += T3_THREADS) ew[w] = __ldg(s + b * wpad + w);
    if (tid == 0) near_s = 0;
    __syncthreads();
    const int SL = N + p.Tg;
    double s1 = 0.0, s2 = 0.0;
    for (int sym = warp; sym < p.S; sym += NW) {
        float2 v[32];
        t4_load_window(rx + b * L, L, SL, (int64_t)sym * SL + p.Tg, 0, false, lane, v);
        t4_pass_a(v, E, fx.tw_t, lane);
        fft32<K2N>(v);
#pragma unroll
        for (int k2 = 0; k2 < K2N; ++k2) E[lane + 32 * k2] = (lane + 32 * k2 < p.Nc) ? v[k2] : make_float2(0.f, 0.f);
        __syncwarp();
        int nears = 0;
        for (int dr = lane; dr < p.Nd; dr += 32) {
            const int c = __ldg(p.data0 + dr);
            // the split chain's equaliser with every desync flag off: G = 1 inside N_carrier, 0 outside
            const float2 e = c < p.Nc ? cmul(E[c], make_float2(1.f, 0.f)) : make_float2(0.f, 0.f);
            float margin = 1.f;
            uint32_t d;                                          // the symbol's bits, first bit in bit 0
            if (QAM16) {
                d = demap16_nib<true>(e.x, e.y, fx.two_a, &margin);
                t4_mer16(e, fx.two_a, a_in, a_out, s1, s2);
            } else {
                const int code = nearest_idx(con, e.x, e.y, &margin);
                const double ir = con.re[code], ii = con.im[code], er = ir - (double)e.x, ei = ii - (double)e.y;
                s1 += ir * ir + ii * ii;
                s2 += er * er + ei * ei;
                d = __brev((uint32_t)code) >> (32 - p.bps);      // demapping.m emits the index MSB first
            }
            nears += margin < near_eps;
            t3_xor_bits(ew, ((int64_t)sym * p.Nd + dr) * p.bps, p.bps, d);
        }
        nears = __reduce_add_sync(0xffffffffu, nears);             // kept in shared memory: one register less across the transform
        if (lane == 0 && nears) atomicAdd(&near_s, nears);
        __syncwarp();                                            // E is the next symbol's transpose tile
    }
    __syncthreads();
    // DeScrambler(d) XOR DeScrambler(s) = e[i] ^ e[i-13] ^ e[i-14], zero history at each frame start
    int errs = 0;
    const int fw = (p.frame_bits + 31) >> 5;
    for (int item = tid; item < p.frames * fw; item += T3_THREADS) {
        const int f = item / fw, wd = item - f * fw;
        const int64_t base = (int64_t)f * p.frame_bits + 32 * wd, end = (int64_t)(f + 1) * p.frame_bits;
        const uint32_t cw = bits_get32(ew, base, end);
        uint32_t o = cw;
        if (p.scramble) {
            const uint32_t prev = wd ? bits_get32(ew, base - 32, end) : 0u;
            o = cw ^ ((cw << 13) | (prev >> 19)) ^ ((cw << 14) | (prev >> 18));
            const int n = min(32, p.frame_bits - 32 * wd);
            if (n < 32) o &= (1u << n) - 1u;
        }
        errs += __popc(o);
    }
    errs = block_sum(errs, red_i);
    s1 = block_sum(s1, red);
    s2 = block_sum(s2, red);
    const int nears = near_s;
    if (tid == 0) {
        mer[b] = s1;
        mer[mer_stride + b] = s2;
        if (errs) atomicAdd(&counts[0], (unsigned long long)errs);
        atomicAdd(&counts[1], (unsigned long long)stream_bits);
        if (nears) atomicAdd(&counts[2], (unsigned long long)nears);
    }
}

static size_t t3_smem(int64_t stream_bits) { return sizeof(float2) * (T3_THREADS / 32) * 32 * T4F_EROW + sizeof(uint32_t) * (size_t)((stream_bits + 31) / 32); }

extern "C" int ofdm_sweep_mer(ofdm_ctx* ctx, const ofdm_link_params* lp, const ofdm_mer_params* mp, double* mer_dev, int64_t* counts_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, lp, "ofdm_sweep_mer: link parameters are NULL");
    REQUIRE(ctx, mp, "ofdm_sweep_mer: MER parameters are NULL");
    REQUIRE(ctx, mer_dev, "ofdm_sweep_mer: mer_dev is NULL");
    REQUIRE(ctx, counts_dev, "ofdm_sweep_mer: counts_dev is NULL");
    if (ctx->precision != OFDM_PREC_F32) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "ofdm_sweep_mer runs the FP32 Task-3 receiver only (context is FP64)");
    if (lp->Nfft != 1024) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "ofdm_sweep_mer supports Nfft = 1024 only (got %d)", lp->Nfft);
    REQUIRE(ctx, mp->n_points > 0, "ofdm_sweep_mer: need at least one point");
    REQUIRE(ctx, mp->constellation_host, "ofdm_sweep_mer: constellation_host is NULL");
    REQUIRE(ctx, mp->snr_db_host, "ofdm_sweep_mer: snr_db_host is NULL");
    REQUIRE(ctx, mp->streams_per_point > 0, "ofdm_sweep_mer: need at least one stream per point");
    REQUIRE(ctx, mp->tile_streams >= 0, "ofdm_sweep_mer: tile_streams must be >= 0 (0 = default)");
    REQUIRE(ctx, mp->world > 0 && mp->rank >= 0 && mp->rank < mp->world, "ofdm_sweep_mer: rank must lie in 0..world-1");
    REQUIRE(ctx, mp->n_taps >= 0 && (mp->n_taps == 0 || mp->taps_host), "ofdm_sweep_mer: bad tap list");
    REQUIRE(ctx, std::isfinite(mp->pilot_scale) && mp->pilot_scale >= 0, "ofdm_sweep_mer: pilot_scale must be finite and >= 0");
    REQUIRE(ctx, mp->pilot_scale > 0 || lp->Np == 0 || lp->pilot_vals_host, "ofdm_sweep_mer: pilot_scale = 0 needs lp->pilot_vals_host");
    REQUIRE(ctx, mp->near_eps >= 0, "ofdm_sweep_mer: near_eps must be >= 0");
    REQUIRE(ctx, lp->S > 0 && lp->SpF > 0 && lp->S % lp->SpF == 0, "ofdm_sweep_mer: S must be a positive multiple of SpF");
    REQUIRE(ctx, lp->N_carrier >= 2 && lp->N_carrier <= lp->Nfft, "ofdm_sweep_mer: N_carrier must lie in 2..Nfft");
    REQUIRE(ctx, lp->Tg >= 0 && lp->Tg <= lp->Nfft, "ofdm_sweep_mer: T_Guard must lie in 0..Nfft");
    REQUIRE(ctx, lp->Np >= 0 && lp->Nd >= 1 && lp->data_carriers_host, "ofdm_sweep_mer: need at least one data carrier");
    const int n_pts = mp->n_points, Nfft = lp->Nfft;
    int bps_max = 0;
    std::vector<ConstTable> ct(n_pts);
    for (int k = 0; k < n_pts; ++k) {
        ct[k] = host_constellation(mp->constellation_host[k]);
        if (ct[k].bps <= 0) return ctx_fail(ctx, OFDM_ERR_INVALID, "ofdm_sweep_mer: point %d has an unknown constellation (%d)", k, mp->constellation_host[k]);
        if (std::isnan(mp->snr_db_host[k])) return ctx_fail(ctx, OFDM_ERR_INVALID, "ofdm_sweep_mer: the SNR of point %d is NaN", k);
        if (mp->nsto_host && mp->nsto_host[k] < 0) return ctx_fail(ctx, OFDM_ERR_INVALID, "ofdm_sweep_mer: the STO of point %d is negative (%d)", k, mp->nsto_host[k]);
        if (mp->cfo_host && !std::isfinite(mp->cfo_host[k])) return ctx_fail(ctx, OFDM_ERR_INVALID, "ofdm_sweep_mer: the CFO of point %d is not finite", k);
        bps_max = std::max(bps_max, ct[k].bps);
    }
    std::vector<int32_t> d0(lp->Nd);
    for (int i = 0; i < lp->Nd; ++i) {
        if (lp->data_carriers_host[i] < 1 || lp->data_carriers_host[i] > Nfft) return ctx_fail(ctx, OFDM_ERR_INVALID, "ofdm_sweep_mer: data carrier out of range");
        // the receiver keeps the N_carrier first bins; Task 3 has no equaliser and decides a carrier past N_carrier from its bin
        if (lp->data_carriers_host[i] > lp->N_carrier)
            return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "ofdm_sweep_mer: a data carrier past N_carrier needs its bin, which the receiver does not keep");
        d0[i] = lp->data_carriers_host[i] - 1;
    }
    const int64_t sym_bits_max = (int64_t)lp->S * lp->Nd * bps_max;
    const size_t smem_max = t3_smem(sym_bits_max);
    if (smem_max > 200 * 1024)
        return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "ofdm_sweep_mer: stream shape needs %zu bytes of shared memory in the receiver (at most 200 KB)", smem_max);
    const int64_t words_max = (sym_bits_max + 31) / 32;
    const int64_t L = (int64_t)lp->S * (Nfft + lp->Tg);

    std::vector<double> h(1, 1.0);                                                  // no multipath: a single unit tap
    if (mp->n_taps > 0)
        REQUIRE(ctx, sweep_dense_taps(mp->taps_host, mp->n_taps, Nfft, h), "ofdm_sweep_mer: tap delays must be integers in [0, Nfft)");
    const int D = (int)h.size();
    std::vector<float> hf(2 * (size_t)D, 0.f);
    for (int d = 0; d < D; ++d) hf[2 * d] = (float)h[d];
    const void* h_dev = ctx_blob(ctx, hf.data(), sizeof(float) * hf.size());
    const int32_t* data0 = (const int32_t*)ctx_blob(ctx, d0.data(), sizeof(int32_t) * d0.size());
    T4FastExtra fx;
    fx.tw_t = (const float2*)t4_twiddle_blob(ctx);
    REQUIRE(ctx, h_dev && data0 && fx.tw_t, "ofdm_sweep_mer: device upload failed");

    SweepTiles tiles(n_pts, mp->streams_per_point, mp->rank, mp->world, mp->tile_streams, 8192);
    if (tiles.count == 0) return OFDM_OK;
    const int64_t tile = tiles.tile;
    auto k13q = rx_t3_kernel<13, true>, k13 = rx_t3_kernel<13, false>, k32q = rx_t3_kernel<32, true>, k32 = rx_t3_kernel<32, false>;
    for (auto f : {k13q, k13, k32q, k32}) CUDA_TRY(ctx, func_smem_optin((const void*)f, (int)smem_max));

    // stream-ordered temporaries, sized for one tile at the largest bps of the call and reused by every tile
    const size_t b_sig = sizeof(float2) * (size_t)L * tile, b_bits = sizeof(uint32_t) * (size_t)(words_max + 1) * tile, b_d = sizeof(double) * tile,
                 b_i = sizeof(int32_t) * tile;
    SweepScratch scr(ctx);
    CUDA_TRY(ctx, scr.alloc({b_sig, b_sig, b_bits, b_bits, b_d, b_d, b_d, b_i}));
    void* tx = scr.get<void>(0);
    void* rx = scr.get<void>(1);
    uint32_t* raw = scr.get<uint32_t>(2);                                            // Philox words s, padded per stream
    uint32_t* sbits = scr.get<uint32_t>(3);                                          // the same bits as one contiguous bitstream
    double* snr_d = scr.get<double>(4);
    double* psum = scr.get<double>(5);
    double* cfo_d = scr.get<double>(6);
    int32_t* sto_d = scr.get<int32_t>(7);

    const int64_t spp = mp->streams_per_point;
    std::vector<double> pv;
    const int rc = tiles.walk([&](int64_t k, int64_t j0, int64_t g, int64_t n) {     // k: point of this tile
        const ConstTable& c = ct[k];
        const int64_t stream_bits = (int64_t)lp->S * lp->Nd * c.bps, words = (stream_bits + 31) / 32;
        ofdm_link_params lp_tx = *lp;                                                // as ofdm_sweep_sync: the TX maps s directly
        lp_tx.constellation = mp->constellation_host[k];
        lp_tx.scramble = 0;
        if (mp->pilot_scale > 0) {                                                   // `Main_model_Task_3.m:57-59`: one real value
            double amax = 0.0;
            for (int i = 0; i < (1 << c.bps); ++i) amax = std::max(amax, std::hypot(c.re[i], c.im[i]));
            pv.assign(2 * (size_t)lp->Np * lp->S, 0.0);
            for (size_t i = 0; i < pv.size(); i += 2) pv[i] = mp->pilot_scale * amax;
            lp_tx.pilot_vals_host = pv.data();
        }
        int rc = ofdm_payload_bits(ctx, raw, n, words, mp->seed, g);
        if (rc) return rc;
        const bool aligned = stream_bits % 32 == 0;
        if (!aligned) ofdm_sweep_pack_bits(ctx, raw, n, words, stream_bits, sbits);
        ofdm_sweep_fill(ctx, n, mp->snr_db_host[k], 1, mp->nsto_host ? mp->nsto_host[k] : 0, mp->cfo_host ? mp->cfo_host[k] : 0.0, snr_d, sto_d, cfo_d);
        // Task 4 order: Noise -> add_STO -> add_CFO -> multipath (`Main_model_Task_4.m:95,103,110,263-264`), one pass
        rc = ofdm_tx_chain_p(ctx, &lp_tx, aligned ? raw : sbits, n, tx, psum);
        if (rc == OFDM_OK) rc = ofdm_channel_t4_p(ctx, tx, n, L, snr_d, psum, nullptr, mp->seed, g, sto_d, cfo_d, Nfft, h_dev, D, rx);
        if (rc) return rc;
        T3Params p;
        p.Tg = lp->Tg; p.Nc = lp->N_carrier; p.S = lp->S; p.Nd = lp->Nd; p.bps = c.bps; p.frame_bits = lp->SpF * lp->Nd * c.bps;
        p.frames = lp->S / lp->SpF; p.scramble = lp->scramble; p.data0 = data0;
        fx.two_a = 2.f * (float)c.re[12];
        const bool q16 = lp_tx.constellation == OFDM_16QAM, small = lp->N_carrier <= 416;
        auto kern = small ? (q16 ? k13q : k13) : (q16 ? k32q : k32);
        // 16QAM: |levels| of the inner and outer points per axis, re = 1 and 3 (`constellation_func.m`)
        kern<<<(unsigned)n, T3_THREADS, t3_smem(stream_bits), ctx->stream>>>(p, fx, make_devconst<float>(lp_tx.constellation), (float)fabs(c.re[12]),
                                                                           (float)fabs(c.re[8]), (const float2*)rx, L, raw, words,
                                                                           mer_dev + k * 2 * spp + j0, spp, (unsigned long long*)(counts_dev + 3 * k),
                                                                           (float)mp->near_eps);
        ctx->launches++;
        return OFDM_OK;
    });
    return scr.finish(rc, "ofdm_sweep_mer launch failed");
}
