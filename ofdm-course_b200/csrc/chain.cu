// Fused link chains, generic-size version: one thread block walks one serial stream.
//   TX: bits -> Scrambler (per-frame reset) -> mapping -> OFDM_map_carriers -> OFDM_modulator
//   RX: OFDM_demodulator -> LS_CE -> equalize_signal -> get_payload -> demapping -> DeScrambler -> BER
// The Nfft = 4096 / N_carrier <= 1024 fast path of the RX chain lives in chain_rx4096.cu.
#include "fft.cuh"
#include "interp.cuh"
#include "fft_reg.cuh"

const void* ofdm_upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex);
#define SLOT_ZERO (-2147483647 - 1)
#define CH_THREADS 256

template <typename T> struct LinkDev {
    int Nfft, logN, Tg, Nc, S, SpF, Nd, Np, bps, scramble;
    int frame_bits, frames;
    uint32_t prev0;
    const int32_t* slot;      // Nfft: data rank / -1-pilot / SLOT_ZERO
    const int32_t* data0;     // Nd 0-based carriers
    const int32_t* pil0;      // Np 0-based carriers
    const cx<T>* pilots;      // Np x S column-major
    const cx<T>* tw;
    DevConst<T> con;
};

struct LinkHost {
    std::vector<int32_t> slot, data0, pil0;
};

uint32_t ofdm_reg_to_prev(const uint8_t* reg) {
    uint32_t p = 0;
    for (int m = 1; m <= 15; ++m) if (reg[m - 1] & 1) p |= 1u << (32 - m);
    return p;
}

template <typename T> static int make_linkdev(ofdm_ctx* ctx, const ofdm_link_params* lp, LinkDev<T>& d) {
    REQUIRE(ctx, lp && lp->Nfft > 0 && is_pow2(lp->Nfft) && lp->S > 0 && lp->SpF > 0 && lp->S % lp->SpF == 0, "bad link parameters (S must be a multiple of SpF)");
    REQUIRE(ctx, lp->Nfft >= 8 && lp->Nfft <= (ctx->precision == OFDM_PREC_F64 ? 4096 : 8192), "unsupported Nfft");
    REQUIRE(ctx, lp->Tg >= 0 && lp->Tg <= lp->Nfft && lp->N_carrier >= 2 && lp->N_carrier <= lp->Nfft, "bad Tg / N_carrier");
    REQUIRE(ctx, lp->Nd >= 1 && lp->Np >= 2 && lp->data_carriers_host && lp->pilot_carriers_host && lp->pilot_vals_host && lp->reg0_host, "missing link tables");
    ConstTable ct = host_constellation(lp->constellation);
    REQUIRE(ctx, ct.bps > 0, "unknown constellation");
    LinkHost h;
    h.slot.assign(lp->Nfft, SLOT_ZERO);
    h.data0.resize(lp->Nd); h.pil0.resize(lp->Np);
    for (int i = 0; i < lp->Nd; ++i) { int c = lp->data_carriers_host[i]; REQUIRE(ctx, c >= 1 && c <= lp->Nfft, "data carrier out of range"); h.slot[c - 1] = i; h.data0[i] = c - 1; }
    for (int i = 0; i < lp->Np; ++i) { int c = lp->pilot_carriers_host[i]; REQUIRE(ctx, c >= 1 && c <= lp->Nfft, "pilot carrier out of range"); h.slot[c - 1] = -1 - i; h.pil0[i] = c - 1; }
    d.Nfft = lp->Nfft; d.logN = ilog2(lp->Nfft); d.Tg = lp->Tg; d.Nc = lp->N_carrier; d.S = lp->S; d.SpF = lp->SpF; d.Nd = lp->Nd; d.Np = lp->Np;
    d.bps = ct.bps; d.scramble = lp->scramble;
    d.frame_bits = lp->SpF * lp->Nd * ct.bps; d.frames = lp->S / lp->SpF;
    d.prev0 = ofdm_reg_to_prev(lp->reg0_host);
    d.slot = (const int32_t*)ctx_blob(ctx, h.slot.data(), sizeof(int32_t) * h.slot.size());
    d.data0 = (const int32_t*)ctx_blob(ctx, h.data0.data(), sizeof(int32_t) * h.data0.size());
    d.pil0 = (const int32_t*)ctx_blob(ctx, h.pil0.data(), sizeof(int32_t) * h.pil0.size());
    d.pilots = (const cx<T>*)ofdm_upload_pilots(ctx, lp->pilot_vals_host, (size_t)lp->Np * lp->S);
    d.tw = (const cx<T>*)ctx_twiddles(ctx, lp->Nfft);
    d.con = make_devconst<T>(lp->constellation);
    REQUIRE(ctx, d.slot && d.data0 && d.pil0 && d.pilots && d.tw, "device upload failed");
    return OFDM_OK;
}

// 32 bits of a shared-memory bit array starting at bit `pos` (words beyond nwords read as 0)
__device__ __forceinline__ uint32_t sm_get32(const uint32_t* w, int pos, int nwords) {
    if (pos < 0) {  // bits before the array read as 0
        if (pos <= -32) return 0u;
        return w[0] << (-pos);
    }
    int wi = pos >> 5, sh = pos & 31;
    uint32_t lo = wi < nwords ? w[wi] : 0u;
    uint32_t hi = (sh && wi + 1 < nwords) ? w[wi + 1] : 0u;
    return __funnelshift_r(lo, hi, sh);
}

// ------------------------------------------------------------------------------------ TX
template <typename T>
__global__ void __launch_bounds__(CH_THREADS) tx_chain_kernel(LinkDev<T> p, const uint32_t* __restrict__ bits, int64_t total_bits, cx<T>* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using C = cx<T>;
    C* a = (C*)smem_raw;
    C* bbuf = a + p.Nfft;
    const int fw = (p.frame_bits + 31) >> 5;
    uint32_t* s0 = (uint32_t*)(bbuf + p.Nfft);
    uint32_t* s1 = s0 + fw;
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x;
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
    for (int f = 0; f < p.frames; ++f) {
        const int64_t base = b * stream_bits + (int64_t)f * p.frame_bits;
        for (int w = tid; w < fw; w += CH_THREADS) {
            uint32_t v = bits_get32(bits, base + 32 * (int64_t)w, min(total_bits, base + p.frame_bits));
            if (w == 0 && p.scramble) v ^= (p.prev0 >> 19) ^ (p.prev0 >> 18);   // fold the register pre-history into the input
            s0[w] = v;
        }
        __syncthreads();
        uint32_t* cur = s0; uint32_t* nxt = s1;
        if (p.scramble) {
            // s = in' * prod_j (1 + x^(13*2^j) + x^(14*2^j)) over GF(2), 13*2^j < frame_bits  (SURVEY KAT 2)
            for (int sh13 = 13, sh14 = 14; sh13 < p.frame_bits; sh13 <<= 1, sh14 <<= 1) {
                for (int w = tid; w < fw; w += CH_THREADS)
                    nxt[w] = cur[w] ^ sm_get32(cur, 32 * w - sh13, fw) ^ sm_get32(cur, 32 * w - sh14, fw);
                __syncthreads();
                uint32_t* t = cur; cur = nxt; nxt = t;
            }
        }
        for (int sf = 0; sf < p.SpF; ++sf) {
            const int s = f * p.SpF + sf;
            for (int k = tid; k < p.Nfft; k += CH_THREADS) {
                int sl = p.slot[k];
                C v = mk<T>(0, 0);
                if (sl >= 0) {
                    int q = sf * p.Nd + sl;                       // QAM symbol number inside the frame
                    uint32_t g = sm_get32(cur, q * p.bps, fw);
                    int idx = 0;
                    for (int i = 0; i < p.bps; ++i) idx = (idx << 1) | ((g >> i) & 1u);
                    v = mk<T>(p.con.re[idx], p.con.im[idx]);
                } else if (sl != SLOT_ZERO) v = p.pilots[(int64_t)s * p.Np + (-1 - sl)];
                a[k] = v;
            }
            __syncthreads();
            C* r = block_fft<T, true>(a, bbuf, p.Nfft, p.logN, p.tw);
            const T scale = (T)1 / (T)p.Nfft;
            C* dst = out + (b * p.S + s) * (int64_t)(p.Nfft + p.Tg);
            for (int i = tid; i < p.Nfft; i += CH_THREADS) {
                C v = cscale(r[i], scale);
                dst[p.Tg + i] = v;
                if (i >= p.Nfft - p.Tg) dst[i - (p.Nfft - p.Tg)] = v;
            }
            __syncthreads();
        }
    }
}

// ---- TX fast path, Nfft = 4096, N_carrier <= 1024, FP32: the modulator's IFFT in registers.
// ifft(X) = conj(fft(conj(X))) / N, and with k = 256 m1 + t only m1 < 4 carries energy (`OFDM_map_carriers.m:3-7` fills
// rows 1..N_carrier), so the forward structure of the RX kernel is reused with the pruning on the INPUT side:
//   pass A  thread t: the four conjugated carriers t + 256 m1 -> 16-point DFT over m1 (12 zero inputs fold away at
//           compile time) x W4096^{t q1} -> [256 q1 + t]
//   pass B  thread (q1, m3): DFT over m2 x W256^{m3 q2} -> [258 q1 + 16 q2 + m3]
//   pass C  thread (q1 = t&15, q2 = t>>4): DFT over m3 -> samples n = t + 256 q3, q3 = 0..15: every store of a warp is
//           one contiguous 256-byte row; rows q3 >= 16 - Tg/256.. also feed the cyclic prefix (`OFDM_modulator.m:7-9`).
// Carriers are built straight into registers from the scrambled frame (shared-memory bit array, log-depth GF(2)
// scrambler as in tx_chain_kernel) -- no frequency grid is ever stored.  Two transform buffers alternate, so a
// symbol costs three block barriers.
#define TXF_XROW 258
#define TXF_XBUF 4128
#define TXF_PAD(fw) ((fw) + ((fw) >> 3) + 2)
__global__ void __launch_bounds__(CH_THREADS, 2) tx4096_kernel(LinkDev<float> p, const uint32_t* __restrict__ bits, int64_t total_bits, float2* __restrict__ out,
                                                               double* __restrict__ power, int64_t B, unsigned long long* __restrict__ next_stream) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* xb = (float2*)smem_raw;                       // two transform buffers
    const int fw = (p.frame_bits + 31) >> 5;
    // two frame bit arrays, each preceded by fw zero words: the scrambler's shifted reads need no range test
    // (pad = fw + fw/8 + 2 words: the x^14 shift of the last doubling reaches 14/13 of a frame back)
    const int pad = TXF_PAD(fw);
    uint32_t* s0 = (uint32_t*)(xb + 2 * TXF_XBUF) + pad;
    uint32_t* s1 = s0 + fw + pad;
    for (int w = threadIdx.x; w < pad; w += CH_THREADS) { s0[w - pad] = 0u; s1[w - pad] = 0u; }
    const int tid = threadIdx.x;
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
    float2 ta[16], tb[16];
#pragma unroll
    for (int q1 = 0; q1 < 16; ++q1) ta[q1] = p.tw[(tid * q1) & 4095];                 // W4096^{t*q1}
    {
        const int m3 = tid & 15;
#pragma unroll
        for (int q2 = 0; q2 < 16; ++q2) {                                             // W256^{m3*q2} / 4096: ifft's 1/N is a power of two,
            const float2 w = p.tw[(16 * m3 * q2) & 4095];                             // so folding it into the twiddle is exact
            tb[q2] = make_float2(w.x * (1.f / 4096.f), w.y * (1.f / 4096.f));
        }
    }
    int slot4[4];
#pragma unroll
    for (int m1 = 0; m1 < 4; ++m1) slot4[m1] = p.slot[tid + 256 * m1];
    int pidx[4];                                          // pilot column row of a pilot carrier (0 otherwise: loaded, not used)
    float2 pv[4];
#pragma unroll
    for (int m1 = 0; m1 < 4; ++m1) {
        pidx[m1] = (slot4[m1] < 0 && slot4[m1] != SLOT_ZERO) ? -1 - slot4[m1] : 0;
        pv[m1] = p.pilots[pidx[m1]];                      // symbol 0
    }
    const bool aligned = (32 % p.bps) == 0;
    __shared__ float2 cs[16];                             // conjugated constellation (a divergent constant-bank index would serialise)
    if (tid < 16) cs[tid] = make_float2(p.con.re[tid], -p.con.im[tid]);
    int par = 0;
    // the payload words of the next frame are requested while the current one is transformed (three per thread cover 24,576-bit frames)
    uint32_t nb[3] = {0u, 0u, 0u};
    auto fetch_frame = [&](int64_t bb, int ff) {
        const int64_t base = bb * stream_bits + (int64_t)ff * p.frame_bits;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const int w = tid + CH_THREADS * j;
            if (w < fw) nb[j] = bits_get32(bits, base + 32 * (int64_t)w, min(total_bits, base + p.frame_bits));
        }
    };
    if ((int64_t)blockIdx.x < B) fetch_frame(blockIdx.x, 0);
    // persistent CTA: the per-thread twiddles, slot roles and the constellation table above are set up once for all its streams
    // With a scheduling counter the CTA's first stream is blockIdx.x and every further one is claimed from the counter (no tail,
    // no lock-step imbalance); the claim is made at the start of the current stream because its last frame already fetches the
    // first frame of the next one.  Two slots by stream parity: the next claim never overwrites a slot still being read.
    __shared__ long long s_next[2];
    int kpar = 0;
    for (int64_t b = blockIdx.x; b < B;) {
        if (next_stream && tid == 0) s_next[kpar] = (long long)gridDim.x + (long long)atomicAdd(next_stream, 1ull);
        int64_t bnext = b + gridDim.x;
        double pacc = 0.0;                                    // this thread's share of sum |x|^2 over the stream, cyclic prefixes included
        for (int f = 0; f < p.frames; ++f) {
            const int64_t base = b * stream_bits + (int64_t)f * p.frame_bits;
            __syncthreads();                                   // previous frame's bit array is no longer read
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int w = tid + CH_THREADS * j;
                if (w < fw) s0[w] = (w == 0 && p.scramble) ? nb[j] ^ (p.prev0 >> 19) ^ (p.prev0 >> 18) : nb[j];   // fold the register pre-history into the input
            }
            for (int w = tid + 3 * CH_THREADS; w < fw; w += CH_THREADS) s0[w] = bits_get32(bits, base + 32 * (int64_t)w, min(total_bits, base + p.frame_bits));
            __syncthreads();
            if (next_stream) bnext = s_next[kpar];            // (written before this frame's barriers)
            if (f + 1 < p.frames) fetch_frame(b, f + 1);
            else if (bnext < B) fetch_frame(bnext, 0);
            uint32_t* cur = s0; uint32_t* nxt = s1;
            if (p.scramble) {
                for (int sh13 = 13, sh14 = 14; sh13 < p.frame_bits; sh13 <<= 1, sh14 <<= 1) {
                    if (((sh13 | sh14) & 31) == 0) {           // from the sixth doubling on both shifts are whole words
                        const int d13 = sh13 >> 5, d14 = sh14 >> 5;
                        for (int w = tid; w < fw; w += CH_THREADS) nxt[w] = cur[w] ^ cur[w - d13] ^ cur[w - d14];
                    } else {                                   // bits [32w - sh, 32w - sh + 32) straddle words w - q - 1 and w - q (sh = 32 q + r); the words before the frame are the zero pad
                        const int q13 = sh13 >> 5, r13 = sh13 & 31, q14 = sh14 >> 5, r14 = sh14 & 31;
                        for (int w = tid; w < fw; w += CH_THREADS) {
                            const int i13 = w - q13, i14 = w - q14;
                            const uint32_t a = __funnelshift_l(cur[i13 - 1], cur[i13], r13);
                            const uint32_t c = __funnelshift_l(cur[i14 - 1], cur[i14], r14);
                            nxt[w] = cur[w] ^ a ^ c;
                        }
                    }
                    __syncthreads();
                    uint32_t* t = cur; cur = nxt; nxt = t;
                }
            }
            for (int sf = 0; sf < p.SpF; ++sf) {
                const int s = f * p.SpF + sf;
                float2* X = xb + par * TXF_XBUF;
                par ^= 1;
                float2 v[16];
                // ---- carriers of this thread, conjugated (mapping.m:14-21, OFDM_map_carriers.m:3-7).  Every lane runs the data path
                // on a clamped slot and picks afterwards: a comb layout mixes data and pilot lanes in every warp.
#pragma unroll
                for (int m1 = 0; m1 < 4; ++m1) {
                    const int sl = slot4[m1];
                    const int qb = (sf * p.Nd + max(sl, 0)) * p.bps;
                    const uint32_t g = aligned ? cur[qb >> 5] >> (qb & 31) : sm_get32(cur, qb, fw);   // bps | 32: a group never straddles a word
                    const float2 cd = cs[__brev(g) >> (32 - p.bps)];      // first bit of the group is the index MSB (`mapping.m:18`, 'left-msb')
                    v[m1] = sl >= 0 ? cd : (sl != SLOT_ZERO ? make_float2(pv[m1].x, -pv[m1].y) : make_float2(0.f, 0.f));
                }
                {                                                         // next symbol's pilot column (the next stream's first), in flight during the transform
                    const int sn = s + 1 < p.S ? s + 1 : 0;
#pragma unroll
                    for (int m1 = 0; m1 < 4; ++m1) pv[m1] = p.pilots[(int64_t)sn * p.Np + pidx[m1]];
                }
                // ---- pass A (rows 4..15 of the column are empty)
                fft16_in4(v);
#pragma unroll
                for (int c = 0; c < 4; ++c)
#pragma unroll
                    for (int d = 0; d < 4; ++d) {
                        const int q1 = c + 4 * d;
                        float2 x = v[4 * c + d];
                        if (q1) x = cmul(x, ta[q1]);
                        X[q1 * 256 + tid] = x;
                    }
                __syncthreads();
                // ---- pass B
                {
                    float2* rp = X + (tid >> 4) * 256 + (tid & 15);
#pragma unroll
                    for (int m2 = 0; m2 < 16; ++m2) v[m2] = rp[16 * m2];
                    __syncthreads();
                    fft16(v);
                    float2* wp = X + (tid >> 4) * TXF_XROW + (tid & 15);
#pragma unroll
                    for (int c = 0; c < 4; ++c)
#pragma unroll
                        for (int d = 0; d < 4; ++d) {
                            const int q2 = c + 4 * d;
                            float2 x = v[4 * c + d];
                            x = q2 ? cmul(x, tb[q2]) : make_float2(x.x * tb[0].x, x.y * tb[0].x);
                            wp[16 * q2] = x;
                        }
                }
                __syncthreads();
                // ---- pass C (all 16 outputs) + conj/N + cyclic prefix
                {
                    const float4* rp = reinterpret_cast<const float4*>(X + (tid & 15) * TXF_XROW + (tid >> 4) * 16);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 w = rp[j];
                        v[2 * j] = make_float2(w.x, w.y);
                        v[2 * j + 1] = make_float2(w.z, w.w);
                    }
                }
                fft16(v);
                float2* dst = out + (b * p.S + s) * (int64_t)(4096 + p.Tg);
                const int cp0 = 4096 - p.Tg;
                float psym = 0.f;
#pragma unroll
                for (int c = 0; c < 4; ++c)
#pragma unroll
                    for (int d = 0; d < 4; ++d) {
                        const int q3 = c + 4 * d;
                        const int n = tid + 256 * q3;
                        const float2 y = make_float2(v[4 * c + d].x, -v[4 * c + d].y);
                        dst[p.Tg + n] = y;
                        if (n >= cp0) dst[n - cp0] = y;
                        const float e = y.x * y.x + y.y * y.y;
                        psym += n >= cp0 ? e + e : e;
                    }
                pacc += (double)psym;
            }
        }
        if (power) {                                           // `Noise.m:3` needs mean |x|^2 of the stream: hand the sum to the channel stage
            __shared__ double red[32];
            const double tot = block_sum(pacc, red);
            if (tid == 0) power[b] = tot;
        }
        b = bnext;
        kpar ^= 1;
    }
}

int ofdm_stream_power_sum(ofdm_ctx* ctx, const void* in, int64_t B, int64_t L, double* power_sum);   // channel.cu
int ofdm_tx1024_fast(ofdm_ctx* ctx, const ofdm_link_params* lp, const uint32_t* bits, int64_t B, void* time, double* power, bool* handled);   // chain_rx_t4.cu
extern "C" int ofdm_tx_chain(ofdm_ctx* ctx, const ofdm_link_params* lp, const uint32_t* bits, int64_t B, void* time) {
    return ofdm_tx_chain_p(ctx, lp, bits, B, time, nullptr);
}
extern "C" int ofdm_tx_chain_p(ofdm_ctx* ctx, const ofdm_link_params* lp, const uint32_t* bits, int64_t B, void* time, double* power) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, bits && time && B >= 0, "bad argument");
    if (B == 0) return OFDM_OK;
    if (ctx->precision == OFDM_PREC_F32 && lp && lp->Nfft == 4096 && lp->N_carrier <= 1024 && !getenv("OFDM_B200_NO_FAST")) {
        LinkDev<float> d;
        int rc = make_linkdev<float>(ctx, lp, d);
        if (rc) return rc;
        bool ok = true;                                   // every occupied row must lie in 1..1024
        for (int i = 0; i < lp->Nd && ok; ++i) ok = lp->data_carriers_host[i] <= 1024;
        for (int i = 0; i < lp->Np && ok; ++i) ok = lp->pilot_carriers_host[i] <= 1024;
        const int fw = (d.frame_bits + 31) / 32;
        const size_t smem = sizeof(float2) * 2 * TXF_XBUF + 2 * sizeof(uint32_t) * (size_t)(fw + TXF_PAD(fw));   // two bit arrays + their zero pads
        if (ok && smem <= 110 * 1024) {
            CUDA_TRY(ctx, func_smem_optin((const void*)tx4096_kernel, (int)smem));
            const int64_t grid = std::min<int64_t>(B, 2 * (int64_t)ctx->sm_count);
            unsigned long long* sched = nullptr;                  // per launch: launches on different streams may overlap
            if (B > grid && !getenv("OFDM_B200_STATIC_STREAMS")) {
                CUDA_TRY(ctx, cudaMallocAsync((void**)&sched, sizeof(unsigned long long), ctx->stream));
                CUDA_TRY(ctx, cudaMemsetAsync(sched, 0, sizeof(unsigned long long), ctx->stream));
            }
            tx4096_kernel<<<(unsigned)grid, CH_THREADS, smem, ctx->stream>>>(d, bits, B * (int64_t)d.frame_bits * d.frames, (float2*)time, power, B, sched);
            if (sched) cudaFreeAsync(sched, ctx->stream);
            LAUNCH_CHECK(ctx);
            return OFDM_OK;
        }
    }
    {
        LinkDev<float> chk;                               // (argument validation is the generic path's)
        bool fast = false;
        if (ctx->precision == OFDM_PREC_F32 && lp && lp->Nfft == 1024) {
            int rc = make_linkdev<float>(ctx, lp, chk);
            if (rc) return rc;
            rc = ofdm_tx1024_fast(ctx, lp, bits, B, time, power, &fast);
            if (rc) return rc;
        }
        if (fast) return OFDM_OK;
    }
    DISPATCH_T(ctx, {
        LinkDev<T> d;
        int rc = make_linkdev<T>(ctx, lp, d);
        if (rc) return rc;
        size_t smem = 2 * sizeof(cx<T>) * d.Nfft + 2 * sizeof(uint32_t) * ((d.frame_bits + 31) / 32);
        auto k = tx_chain_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<(unsigned)B, CH_THREADS, smem, ctx->stream>>>(d, bits, B * (int64_t)d.frame_bits * d.frames, (cx<T>*)time);
    });
    LAUNCH_CHECK(ctx);
    if (power) return ofdm_stream_power_sum(ctx, time, B, (int64_t)lp->S * (lp->Nfft + lp->Tg), power);   // generic shapes: separate pass
    return OFDM_OK;
}

// ------------------------------------------------------------------------------------ RX (generic)
template <typename T>
__global__ void __launch_bounds__(CH_THREADS) rx_chain_kernel(LinkDev<T> p, PlanDev<T> plan, const cx<T>* __restrict__ rx, const uint32_t* __restrict__ txbits,
                                                              int64_t total_bits, uint32_t* __restrict__ outbits, cx<T>* __restrict__ Hout,
                                                              unsigned long long* __restrict__ counts, int32_t* __restrict__ err_stream, T near_eps) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using C = cx<T>;
    __shared__ int red_i[32];
    C* a = (C*)smem_raw;
    C* bbuf = a + p.Nfft;
    C* y = bbuf + p.Nfft;
    C* dk = y + plan.n_knots;
    C* Hs = dk + plan.n_knots;                       // Nc
    const int fw = (p.frame_bits + 31) >> 5;
    uint32_t* raw = (uint32_t*)(Hs + p.Nc);          // fw words of demapped bits
    uint8_t* symidx = (uint8_t*)(raw + fw);          // SpF*Nd decided constellation indices of the frame
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x;
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
    int errs = 0, nears = 0;
    for (int s = 0; s < p.S; ++s) {
        const C* src = rx + (b * p.S + s) * (int64_t)(p.Nfft + p.Tg) + p.Tg;
        for (int i = tid; i < p.Nfft; i += CH_THREADS) a[i] = src[i];
        __syncthreads();
        C* r = block_fft<T, false>(a, bbuf, p.Nfft, p.logN, p.tw);
        if (s == 0) {   // LS_CE: first symbol only (`LS_CE.m:27-31`)
            for (int k = tid; k < p.Np; k += CH_THREADS) y[plan.ext_lo + k] = cdiv(r[p.pil0[k]], p.pilots[k]);
            __syncthreads();
            plan_apply(plan, y, dk, Hs);
            __syncthreads();
            if (Hout) for (int k = tid; k < p.Nc; k += CH_THREADS) Hout[b * p.Nc + k] = Hs[k];
        }
        const int sf = s % p.SpF;
        for (int dr = tid; dr < p.Nd; dr += CH_THREADS) {   // equalize_signal + get_payload + demapping decision
            int c = p.data0[dr];
            C e = (c < p.Nc) ? cdiv(r[c], Hs[c]) : mk<T>(0, 0);   // rows beyond N_carrier are zeros (`equalize_signal.m:3`)
            T margin;
            int idx = nearest_idx(p.con, e.x, e.y, &margin);
            if (margin < near_eps) ++nears;
            symidx[sf * p.Nd + dr] = (uint8_t)idx;
        }
        __syncthreads();
        if (sf == p.SpF - 1) {   // frame complete: pack bits, DeScrambler, compare
            const int f = s / p.SpF;
            for (int w = tid; w < fw; w += CH_THREADS) {
                const int b0 = 32 * w, b1 = min(b0 + 32, p.frame_bits);
                uint32_t word = 0;
                for (int q = b0 / p.bps; q * p.bps < b1; ++q) {
                    int idx = symidx[q];
                    for (int i = 0; i < p.bps; ++i) {
                        int pos = q * p.bps + i;
                        if (pos >= b0 && pos < b1 && ((idx >> (p.bps - 1 - i)) & 1)) word |= 1u << (pos - b0);
                    }
                }
                raw[w] = word;
            }
            __syncthreads();
            const int64_t base = b * stream_bits + (int64_t)f * p.frame_bits;
            for (int w = tid; w < fw; w += CH_THREADS) {
                uint32_t cur = raw[w];
                uint32_t o = cur;
                if (p.scramble) {
                    uint32_t prev = w ? raw[w - 1] : p.prev0;
                    o = cur ^ ((cur << 13) | (prev >> 19)) ^ ((cur << 14) | (prev >> 18));
                }
                const int n = min(32, p.frame_bits - 32 * w);
                if (n < 32) o &= (1u << n) - 1u;
                if (txbits) {
                    uint32_t t = bits_get32(txbits, base + 32 * (int64_t)w, min(total_bits, base + p.frame_bits));
                    errs += __popc(o ^ t);
                }
                if (outbits) bits_put(outbits, base + 32 * (int64_t)w, n, o);
            }
            __syncthreads();
        }
    }
    errs = block_sum(errs, red_i);
    nears = block_sum(nears, red_i);
    if (tid == 0) {
        if (counts) {
            if (errs) atomicAdd(&counts[0], (unsigned long long)errs);
            atomicAdd(&counts[1], (unsigned long long)stream_bits);
            if (nears) atomicAdd(&counts[2], (unsigned long long)nears);
        }
        if (err_stream) err_stream[b] = errs;
    }
}

int ofdm_rx_chain_fast4096(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx, int64_t B, const uint32_t* tx_bits, uint32_t* out_bits,
                           void* H, int64_t* counts, int32_t* err_stream, double near_eps, bool* handled);

extern "C" int ofdm_rx_chain_t5(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx, int64_t B, const uint32_t* tx_bits, uint32_t* out_bits,
                                void* H, int64_t* counts, int32_t* err_stream, double near_eps) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, rx && B >= 0 && lp, "bad argument");
    if (B == 0) return OFDM_OK;
    bool handled = false;
    int rc = ofdm_rx_chain_fast4096(ctx, lp, rx, B, tx_bits, out_bits, H, counts, err_stream, near_eps, &handled);
    if (rc || handled) return rc;
    DISPATCH_T(ctx, {
        LinkDev<T> d;
        rc = make_linkdev<T>(ctx, lp, d);
        if (rc) return rc;
        const InterpPlan* pl = ctx_plan(ctx, lp->pilot_carriers_host, lp->Np, lp->N_carrier, nullptr, lp->N_carrier, OFDM_INTERP_SPLINE);
        REQUIRE(ctx, pl != nullptr, "plan construction failed");
        for (int i = 0; i < lp->Np; ++i) REQUIRE(ctx, lp->pilot_carriers_host[i] <= lp->N_carrier, "pilot beyond N_carrier");
        const int64_t stream_bits = (int64_t)d.frame_bits * d.frames;
        if (out_bits && (stream_bits % 32 != 0 || d.frame_bits % 32 != 0))
            CUDA_TRY(ctx, cudaMemsetAsync(out_bits, 0, sizeof(uint32_t) * OFDM_BIT_WORDS(B * stream_bits), ctx->stream));
        const int fw = (d.frame_bits + 31) / 32;
        size_t smem = sizeof(cx<T>) * (2 * (size_t)d.Nfft + 2 * (size_t)pl->n_knots + d.Nc) + sizeof(uint32_t) * fw + (size_t)d.SpF * d.Nd + 16;
        auto k = rx_chain_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k, (int)smem));
        k<<<(unsigned)B, CH_THREADS, smem, ctx->stream>>>(d, plan_dev<T>(pl), (const cx<T>*)rx, tx_bits, B * stream_bits, out_bits, (cx<T>*)H,
                                                           (unsigned long long*)counts, err_stream, (T)near_eps);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// ------------------------------------------------------------------------------------ RX from host buffers
extern "C" int ofdm_rx_chain_t5_host(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx_host, int64_t B, const uint32_t* tx_bits_host,
                                     uint32_t* out_bits_host, void* H_host, int64_t* counts_host, int64_t chunk) {
    return ofdm_rx_chain_t5_host_eps(ctx, lp, rx_host, B, tx_bits_host, out_bits_host, H_host, counts_host, chunk, 0.0);
}

extern "C" int ofdm_rx_chain_t5_host_eps(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx_host, int64_t B, const uint32_t* tx_bits_host,
                                         uint32_t* out_bits_host, void* H_host, int64_t* counts_host, int64_t chunk, double near_eps) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, rx_host && lp && B >= 0 && counts_host, "bad argument");
    ConstTable ct = host_constellation(lp->constellation);
    REQUIRE(ctx, ct.bps > 0, "unknown constellation");
    const size_t esz = ctx->precision == OFDM_PREC_F64 ? sizeof(double2) : sizeof(float2);
    const int64_t stream_bits = (int64_t)lp->S * lp->Nd * ct.bps;
    REQUIRE(ctx, stream_bits % 32 == 0, "host-buffer chain needs word-aligned streams (stream bits % 32 == 0)");
    const int64_t words = stream_bits / 32;
    const int64_t L = (int64_t)lp->S * (lp->Nfft + lp->Tg);
    if (chunk <= 0) chunk = 2048;
    chunk = std::min<int64_t>(chunk, std::max<int64_t>(B, 1));
    // per-slot device staging: rx | tx bits | out bits | H
    // the cyclic prefix is never consumed by this chain: a strided copy leaves it on the host (-11% PCIe bytes)
    ofdm_link_params lpd = *lp;
    lpd.Tg = 0;
    const int64_t Ld = (int64_t)lp->S * lp->Nfft;
    const size_t rx_b = esz * Ld * chunk, bits_b = sizeof(uint32_t) * words * chunk, H_b = esz * lp->N_carrier * chunk;
    const size_t slot_b = rx_b + 2 * bits_b + H_b + 256;
    if (ctx->staging_bytes < slot_b) {
        for (int i = 0; i < 2; ++i) { if (ctx->staging[i]) cudaFree(ctx->staging[i]); ctx->staging[i] = nullptr; }
        for (int i = 0; i < 2; ++i) CUDA_TRY(ctx, cudaMalloc(&ctx->staging[i], slot_b));
        ctx->staging_bytes = slot_b;
    }
    // the three counters live in the context (allocated once): no cudaMalloc/cudaFree, both device-synchronising, per call
    if (!ctx->host_counts_d) {
        CUDA_TRY(ctx, cudaMalloc((void**)&ctx->host_counts_d, 64));
        ctx->owned.push_back(ctx->host_counts_d);
    }
    int64_t* counts_d = ctx->host_counts_d;
    cudaStream_t user = ctx->stream;
    cudaEvent_t done[2] = {ctx->ev[0], ctx->ev[1]};
    int rc = OFDM_OK;
    // one exit path: CUDA failures inside the chunk loop fall through to the drain below instead of returning with copies in flight
#define HOST_TRY(expr)                                                                                                              \
    do {                                                                                                                            \
        cudaError_t _e = (expr);                                                                                                    \
        if (_e != cudaSuccess && rc == OFDM_OK) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
    HOST_TRY(cudaMemsetAsync(counts_d, 0, 3 * sizeof(int64_t), user));
    HOST_TRY(cudaEventRecord(ctx->ev[2], user));
    for (int i = 0; i < 2; ++i) HOST_TRY(cudaStreamWaitEvent(ctx->copy_stream[i], ctx->ev[2], 0));
    for (int64_t c0 = 0, it = 0; c0 < B && rc == OFDM_OK; c0 += chunk, ++it) {
        const int slot = (int)(it & 1);
        const int64_t nb = std::min(chunk, B - c0);
        cudaStream_t st = ctx->copy_stream[slot];   // each slot is a self-contained in-order pipeline: H2D -> kernel -> D2H
        unsigned char* base = (unsigned char*)ctx->staging[slot];
        void* rx_d = base;
        uint32_t* tx_d = (uint32_t*)(base + rx_b);
        uint32_t* ob_d = (uint32_t*)(base + rx_b + bits_b);
        void* H_d = base + rx_b + 2 * bits_b;
        HOST_TRY(cudaMemcpy2DAsync(rx_d, esz * lp->Nfft, (const unsigned char*)rx_host + esz * (L * c0 + lp->Tg), esz * (lp->Nfft + lp->Tg), esz * lp->Nfft,
                                   (size_t)nb * lp->S, cudaMemcpyHostToDevice, st));
        if (tx_bits_host) HOST_TRY(cudaMemcpyAsync(tx_d, tx_bits_host + words * c0, sizeof(uint32_t) * words * nb, cudaMemcpyHostToDevice, st));
        if (rc) break;
        ctx->stream = st;
        rc = ofdm_rx_chain_t5(ctx, &lpd, rx_d, nb, tx_bits_host ? tx_d : nullptr, out_bits_host ? ob_d : nullptr, H_host ? H_d : nullptr, counts_d, nullptr, near_eps);
        ctx->stream = user;
        if (rc) break;
        if (out_bits_host) HOST_TRY(cudaMemcpyAsync(out_bits_host + words * c0, ob_d, sizeof(uint32_t) * words * nb, cudaMemcpyDeviceToHost, st));
        if (H_host) HOST_TRY(cudaMemcpyAsync((unsigned char*)H_host + esz * lp->N_carrier * c0, H_d, esz * lp->N_carrier * nb, cudaMemcpyDeviceToHost, st));
        HOST_TRY(cudaEventRecord(done[slot], st));
    }
    // join: slot 1 waits for slot 0, reads the counters back, and the host waits for slot 1 only
    if (rc == OFDM_OK) {
        HOST_TRY(cudaEventRecord(done[0], ctx->copy_stream[0]));
        HOST_TRY(cudaStreamWaitEvent(ctx->copy_stream[1], done[0], 0));
        HOST_TRY(cudaMemcpyAsync(counts_host, counts_d, 3 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->copy_stream[1]));
    }
    for (int i = 0; i < 2; ++i) HOST_TRY(cudaStreamSynchronize(ctx->copy_stream[i]));
#undef HOST_TRY
    return rc;
}
