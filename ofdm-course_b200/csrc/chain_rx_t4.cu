// Fused Task-4 RX chain (SURVEY M2, `Task 4/Main_model_Task_4.m:277-366`), FP32, one persistent CTA per stream:
//   AutoCorrFunction (sync.cu, one pass)  ->  this kernel:
//   add_STO(TgPosition), add_STO(-(Nfft+Tg))      as an index offset + zero fill on load      [add_STO.m:5-9]
//   add_CFO(-FreqOffset), remove_IFO              as ONE rotation exp(-2j*pi*(FFO+IFO)*n/Nfft) [add_CFO.m:6-7, remove_IFO.m:5-9]
//   OFDM_demodulator                              shared-memory Stockham FFT per symbol        [OFDM_demodulator.m:5-8]
//   fine_sync                                     estimators in double on the pilots           [Task 4/fine_sync.m:25-58]
//   estimate_channel + equalize_signal            symbol-averaged pilot LS, not-a-knot spline  [estimate_channel.m:4-8, equalize_signal.m:6]
//   get_payload, demapping, DeScrambler, BER      per 5-symbol frame (frames are not word aligned: 6,640 bits)
// The N_carrier useful bins of every symbol are parked in a per-CTA global scratch (stays in L2) between the
// FFT phase and the decision phase, because fine_sync's estimates need all symbols before any of them is corrected.
#include "fft.cuh"
#include "interp.cuh"
#include "fft_reg.cuh"

const void* ofdm_upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex);
uint32_t ofdm_reg_to_prev(const uint8_t* reg);
#define T4_THREADS 256
#define SLOT_ZERO (-2147483647 - 1)

struct T4Params {
    int Nfft, logN, Tg, Nc, S, SpF, Nd, Np, bps, scramble, frame_bits, frames;
    int time_desync, freq_desync, mp_desync;
    uint32_t prev0;
    const int32_t* data0;      // Nd 0-based data carriers
    const int32_t* pil0;       // Np 0-based pilot carriers
    const float2* pilots;      // Np x S column-major (float)
    const double2* pilots_d;   // same in double for the estimators
    const float2* tw;          // W_Nfft^k
};

__device__ __forceinline__ float2 rot_from_cycles(double cyc) {   // exp(-2j*pi*cyc), range-reduced in double
    double fr = cyc - floor(cyc);
    float s, c;
    sincospif((float)(-2.0 * fr), &s, &c);
    return make_float2(c, s);
}

__global__ void __launch_bounds__(T4_THREADS) rx_t4_kernel(T4Params p, PlanDev<float> plan, DevConst<float> con, const float2* __restrict__ rx, int64_t B,
                                                           int64_t L, const int32_t* __restrict__ tg_pos, const double* __restrict__ freq_off,
                                                           float2* __restrict__ scratch, const uint32_t* __restrict__ txbits, int64_t total_bits,
                                                           uint32_t* __restrict__ outbits, unsigned long long* __restrict__ counts,
                                                           int32_t* __restrict__ ifo_out, double* __restrict__ tau_out, double* __restrict__ phase_out,
                                                           float2* __restrict__ Hout, float near_eps) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double red[32];
    __shared__ int red_i[32];
    __shared__ int cnt[T4_THREADS];
    float2* fa = (float2*)smem_raw;                 // FFT ping-pong
    float2* fb = fa + p.Nfft;
    float2* Yp = fb + p.Nfft;                       // pilots of every symbol, [s][p]
    float2* rot_s = Yp + p.S * p.Np;                // per-symbol base rotation
    float2* G = rot_s + p.S;                        // per-carrier correction / equaliser, Nc
    float2* yk = G + p.Nc;                          // spline knots
    float2* dk = yk + plan.n_knots;
    double* taus = (double*)(dk + plan.n_knots);    // Np*S differential timing estimates
    uint32_t* raw = (uint32_t*)(taus + p.S * p.Np); // frame words
    const int fw = (p.frame_bits + 31) >> 5;
    uint8_t* symidx = (uint8_t*)(raw + fw);         // SpF * Nd decisions
    const int tid = threadIdx.x;
    const int SL = p.Nfft + p.Tg;
    const int M = p.Np * p.S;
    float2* Ysc = scratch + (int64_t)blockIdx.x * p.S * p.Nc;   // this CTA's parking area
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
    const int NJ = p.Nfft / T4_THREADS;             // samples per thread per symbol (Nfft >= 256)

    for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
        const float2* r = rx + b * L;
        const int tg = p.time_desync ? tg_pos[b] : 0;
        const double fo = p.freq_desync ? freq_off[b] : 0.0;
        // sample n of the time-corrected stream (`Main_model_Task_4.m:292-294`)
        auto sample = [&](int64_t n) -> float2 {
            if (!p.time_desync) return r[n];
            int64_t m = n - SL + tg;
            return (n >= SL && m < L && m >= 0) ? r[m] : make_float2(0.f, 0.f);
        };
        // ---- remove_IFO: first bin of |fft(y3(Nfft+1:2*Nfft))| above 0.77 (`remove_IFO.m:5-8`)
        int ifo = 0;
        if (p.freq_desync) {
            for (int i = tid; i < p.Nfft; i += T4_THREADS) {
                const int64_t n = p.Nfft + i;
                fa[i] = cmul(sample(n), rot_from_cycles(fo * (double)n / p.Nfft));
            }
            __syncthreads();
            float2* X = block_fft<float, false>(fa, fb, p.Nfft, p.logN, p.tw);
            int first = 0x7fffffff;
            for (int i = tid; i < p.Nfft; i += T4_THREADS) {
                double re = X[i].x, im = X[i].y;
                if (sqrt(re * re + im * im) > 0.77) { first = i; break; }
            }
            first = block_min(first, red_i);
            ifo = (first == 0x7fffffff) ? -1 : first;
            __syncthreads();
        }
        if (tid == 0 && ifo_out) ifo_out[b] = ifo;
        const double c = fo + (ifo > 0 ? ifo : 0);   // total derotation in cycles per Nfft samples
        float2 w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) if (j < NJ) w[j] = rot_from_cycles(c * (double)(tid + T4_THREADS * j) / p.Nfft);
        for (int s = tid; s < p.S; s += T4_THREADS) rot_s[s] = rot_from_cycles(c * (double)((int64_t)s * SL + p.Tg) / p.Nfft);
        __syncthreads();
        // ---- OFDM_demodulator for every symbol; park the useful bins, keep the pilots
        for (int s = 0; s < p.S; ++s) {
            const int64_t n0 = (int64_t)s * SL + p.Tg;
            const float2 rs = rot_s[s];
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (j < NJ) {
                    const int i = tid + T4_THREADS * j;
                    float2 x = sample(n0 + i);
                    if (p.freq_desync) x = cmul(x, cmul(rs, w[j]));
                    fa[i] = x;
                }
            __syncthreads();
            float2* X = block_fft<float, false>(fa, fb, p.Nfft, p.logN, p.tw);
            for (int k = tid; k < p.Nc; k += T4_THREADS) Ysc[(int64_t)s * p.Nc + k] = X[k];
            for (int q = tid; q < p.Np; q += T4_THREADS) Yp[s * p.Np + q] = X[p.pil0[q]];
            __syncthreads();
        }
        // ---- fine_sync estimators (`Task 4/fine_sync.m:25-35,47-52`), in double
        double tau = 0.0, phase = 0.0;
        if (p.time_desync || p.freq_desync) {
            const double deltak = (double)(p.pil0[1] - p.pil0[0]);
            auto q_at = [&](int i) -> double2 { return cmulc(p.pilots_d[i], to_d(Yp[i])); };   // tx * conj(rx), flat column-major index
            auto tau_at = [&](int j) -> double { double2 d = cmulc(q_at(j + 1), q_at(j)); return atan2(d.y, d.x) / (2.0 * CUDART_PI * deltak); };
            const int n = M - 1;
            for (int j = tid; j < n; j += T4_THREADS) taus[j] = tau_at(j);                  // taus(j+1) of the reference (:25-30)
            __syncthreads();
            // mask = [false, abs(diffs)<1e-3 & abs(diffs)~=0]; taus_result = taus(mask); mean(taus_result(Np+1:end))  (:32-35)
            const int CH = (n + T4_THREADS - 1) / T4_THREADS;
            const int lo = min(tid * CH, n), hi = min(lo + CH, n);
            int cmask = 0;
            for (int j = max(lo, 1); j < hi; ++j) { double d = fabs(taus[j] - taus[j - 1]); cmask += (d < 1e-3 && d != 0.0); }
            int rank = block_exclusive_scan(cmask, red_i);      // survivors before this thread's chunk
            double sum = 0; int kept = 0;
            for (int j = max(lo, 1); j < hi; ++j) {
                double d = fabs(taus[j] - taus[j - 1]);
                if (d < 1e-3 && d != 0.0) { if (rank >= p.Np) { sum += taus[j]; ++kept; } ++rank; }
            }
            sum = block_sum(sum, red);
            double nk = block_sum((double)kept, red);
            tau = sum / nk;
            double ps = 0; int pn = 0;
            for (int i = tid; i < M; i += T4_THREADS) {
                const int pq = i % p.Np;
                double2 rxv = to_d(Yp[i]);
                if (p.time_desync) { double sn, cs; sincospi(2.0 * tau * (double)p.pil0[pq], &sn, &cs); rxv = cmul(rxv, make_double2(cs, sn)); }
                double2 qq = cmulc(p.pilots_d[i], rxv);
                double a = atan2(qq.y, qq.x);
                if (fabs(a) > 1e-3) { ps += a; ++pn; }
            }
            ps = block_sum(ps, red);
            double pk = block_sum((double)pn, red);
            phase = ps / pk;
            if (tid == 0) { if (tau_out) tau_out[b] = tau; if (phase_out) phase_out[b] = phase; }
        }
        // ---- per-carrier correction factor exp(j*(2*pi*tau*k*[time] + phase*[freq])) (`fine_sync.m:38-58`)
        for (int k = tid; k < p.Nc; k += T4_THREADS) {
            double sn = 0.0, cs = 1.0;
            if (p.time_desync || p.freq_desync) {
                double ang = (p.time_desync ? 2.0 * tau * (double)k : 0.0);     // in units of pi
                double s1, c1, s2 = 0.0, c2 = 1.0;
                sincospi(ang, &s1, &c1);
                if (p.freq_desync) sincos(phase, &s2, &c2);
                cs = c1 * c2 - s1 * s2; sn = s1 * c2 + c1 * s2;
            }
            G[k] = make_float2((float)cs, (float)sn);
        }
        __syncthreads();
        // ---- estimate_channel on the corrected grid + equalize_signal (`estimate_channel.m:4-8`)
        if (p.mp_desync) {
            for (int q = tid; q < p.Np; q += T4_THREADS) {
                float sr = 0.f, si = 0.f;
                const float2 g = G[p.pil0[q]];
                for (int s = 0; s < p.S; ++s) { float2 v = cdiv(cmul(Yp[s * p.Np + q], g), p.pilots[(int64_t)s * p.Np + q]); sr += v.x; si += v.y; }
                yk[q] = make_float2(sr / (float)p.S, si / (float)p.S);
            }
            __syncthreads();
            float2* Hrow = Hout ? Hout + b * p.Nc : nullptr;
            plan_apply_fn<float>(plan, yk, dk, [&](int k, float2 h) {
                if (Hrow) Hrow[k] = h;
                G[k] = cdiv(G[k], h);            // equalised = Y * cf / H
            });
            __syncthreads();
        }
        // ---- get_payload, demapping, DeScrambler, BER
        int errs = 0, nears = 0;
        for (int s = 0; s < p.S; ++s) {
            const int sf = s % p.SpF;
            for (int dr = tid; dr < p.Nd; dr += T4_THREADS) {
                const int cidx = p.data0[dr];
                float2 e = (cidx < p.Nc) ? cmul(Ysc[(int64_t)s * p.Nc + cidx], G[cidx]) : make_float2(0.f, 0.f);
                float margin;
                int idx = nearest_idx(con, e.x, e.y, &margin);
                if (margin < near_eps) ++nears;
                symidx[sf * p.Nd + dr] = (uint8_t)idx;
            }
            __syncthreads();
            if (sf == p.SpF - 1) {
                const int f = s / p.SpF;
                for (int wd = tid; wd < fw; wd += T4_THREADS) {
                    const int b0 = 32 * wd, b1 = min(b0 + 32, p.frame_bits);
                    uint32_t word = 0;
                    for (int q = b0 / p.bps; q * p.bps < b1; ++q) {
                        int idx = symidx[q];
                        for (int i = 0; i < p.bps; ++i) {
                            int pos = q * p.bps + i;
                            if (pos >= b0 && pos < b1 && ((idx >> (p.bps - 1 - i)) & 1)) word |= 1u << (pos - b0);
                        }
                    }
                    raw[wd] = word;
                }
                __syncthreads();
                const int64_t base = b * stream_bits + (int64_t)f * p.frame_bits;
                for (int wd = tid; wd < fw; wd += T4_THREADS) {
                    uint32_t cw = raw[wd], o = cw;
                    if (p.scramble) {
                        uint32_t prev = wd ? raw[wd - 1] : p.prev0;
                        o = cw ^ ((cw << 13) | (prev >> 19)) ^ ((cw << 14) | (prev >> 18));
                    }
                    const int n = min(32, p.frame_bits - 32 * wd);
                    if (n < 32) o &= (1u << n) - 1u;
                    if (txbits) errs += __popc(o ^ bits_get32(txbits, base + 32 * (int64_t)wd, min(total_bits, base + p.frame_bits)));
                    if (outbits) bits_put(outbits, base + 32 * (int64_t)wd, n, o);
                }
                __syncthreads();
            }
        }
        errs = block_sum(errs, red_i);
        nears = block_sum(nears, red_i);
        if (tid == 0 && counts) {
            if (errs) atomicAdd(&counts[0], (unsigned long long)errs);
            atomicAdd(&counts[1], (unsigned long long)stream_bits);
            if (nears) atomicAdd(&counts[2], (unsigned long long)nears);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------
// Fast path for Nfft = 1024 (the Task-4 shape): same chain, same order of operations, but
//   * a symbol is transformed by ONE WARP: 1024 = 32 x 32, lane n2 runs a register-resident 32-point DFT over
//     n1 (x[32 n1 + n2], coalesced 256-byte rows straight from global memory, all 32 loads in flight), the
//     W1024^{n2 k1} twiddles come from a transposed table (L1-resident), a 32 x 33 warp-private shared tile does
//     the transpose, lane k1 runs the second 32-point DFT over n2 and keeps bins k1 + 32 k2 -- only k2 < K2N
//     (N_carrier <= 32 K2N) are ever produced, the rest is pruned at compile time.  No block barrier inside the
//     symbol loop: the eight warps of a CTA work on eight symbols of the stream at once.
//   * the per-symbol base rotation of the CFO/IFO removal is applied to the kept bins (the DFT is linear), the
//     per-sample part exp(-2j*pi*c*i/Nfft) comes from a per-stream shared table;
//   * 16QAM decisions use the separable rule and the frame's bits are packed eight symbols per word.
// Estimators (fine_sync) and the channel estimate are the code of the generic kernel above.
#define T4F_EROW 33
__device__ __forceinline__ float2 ldg_stream(const float2* p) {   // the sample stream is read once here: keep it out of L1 (tables live there)
    float2 r;
    asm("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
struct T4FastExtra {
    const float2* tw_t;        // [k1][n2] = W1024^{n2*k1}: transposed twiddles, coalesced across lanes
    float two_a;
};

template <int K2N, bool QAM16, bool NEAR>
__global__ void __launch_bounds__(T4_THREADS, 2) rx_t4_fast_kernel(T4Params p, T4FastExtra fx, PlanDev<float> plan, DevConst<float> con,
                                                                    const float2* __restrict__ rx, int64_t B, int64_t L,
                                                                    const int32_t* __restrict__ tg_pos, const double* __restrict__ freq_off,
                                                                    float2* __restrict__ scratch, const uint32_t* __restrict__ txbits, int64_t total_bits,
                                                                    uint32_t* __restrict__ outbits, unsigned long long* __restrict__ counts,
                                                                    int32_t* __restrict__ ifo_out, double* __restrict__ tau_out,
                                                                    double* __restrict__ phase_out, float2* __restrict__ Hout, float near_eps) {
    constexpr int N = 1024;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double red[32];
    __shared__ int red_i[32];
    __shared__ int cnt[T4_THREADS];
    __shared__ int ifo_s, next_sym;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = T4_THREADS / 32;
    const int M = p.Np * p.S;
    // layout: [phase-1 tiles | phase-2 taus | phase-3 decisions] (aliased), wtab, Yp, rot_s, G, yk, dk
    const size_t tiles_bytes = sizeof(float2) * (size_t)NW * 32 * T4F_EROW;
    const size_t taus_bytes = sizeof(double) * (size_t)M;
    float2* tiles = (float2*)smem_raw;
    double* taus = (double*)smem_raw;
    float2* wtab = (float2*)(smem_raw + ((tiles_bytes > taus_bytes ? tiles_bytes : taus_bytes) + 15) / 16 * 16);
    float2* Yp = wtab + N;                           // pilots of every symbol, [s][p]
    float2* rot_s = Yp + M;                          // per-symbol base rotation
    float2* G = rot_s + p.S;                         // per-carrier correction / equaliser, Nc
    float2* yk = G + p.Nc;
    float2* dk = yk + plan.n_knots;
    const int fw = (p.frame_bits + 31) >> 5;
    float2* E = tiles + warp * 32 * T4F_EROW;        // this warp's transpose tile
    const int SL = N + p.Tg;
    float2* Ysc = scratch + (int64_t)blockIdx.x * p.S * p.Nc;   // this CTA's parking area (stays in L2)
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;

    // one symbol-sized window starting at stream sample n0 (after the two add_STO calls): DFT bins k < 32*KK
    // X[lane + 32 k2] are returned in v[k2]; `derot` multiplies sample i by wtab[i] first.
    auto load_window = [&](const float2* r, int64_t n0, int tg, bool tshift, float2* v) {
        // sample n of the corrected stream is r[n - SL + tg] for n >= SL inside the record, else 0 (`add_STO.m:5-9`)
        const int64_t m0 = tshift ? n0 - SL + tg : n0;
        const bool all_in = (m0 >= 0 && m0 + N <= L && (!tshift || n0 >= SL));
        if (all_in) {
            const float2* q = r + m0 + lane;
#pragma unroll
            for (int n1 = 0; n1 < 32; ++n1) v[n1] = ldg_stream(q + 32 * n1);
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; ++n1) {
                const int64_t m = m0 + 32 * n1 + lane;
                const bool ok = m >= 0 && m < L && (!tshift || n0 + 32 * n1 + lane >= SL);
                v[n1] = ok ? ldg_stream(r + m) : make_float2(0.f, 0.f);
            }
        }
    };
    auto pass_a = [&](float2* v) {      // DFT over n1, twiddle, transpose through the tile
        fft32<32>(v);
#pragma unroll
        for (int k1 = 0; k1 < 32; ++k1) {
            float2 x = v[k1];
            if (k1) x = cmul(x, __ldg(fx.tw_t + 32 * k1 + lane));
            E[k1 * T4F_EROW + lane] = x;
        }
        __syncwarp();
#pragma unroll
        for (int n2 = 0; n2 < 32; ++n2) v[n2] = E[lane * T4F_EROW + n2];
        __syncwarp();
    };

    for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
        const float2* r = rx + b * L;
        const int tg = p.time_desync ? tg_pos[b] : 0;
        const double fo = p.freq_desync ? freq_off[b] : 0.0;
        const bool tshift = p.time_desync != 0;
        // ---- remove_IFO (`remove_IFO.m:5-8`) overlapped with the first round of symbols.
        // Derotating by c = fo + ifo cycles per Nfft samples is derotating by fo, shifting the spectrum by ifo bins and
        // a per-symbol phase: X_c[k] = exp(-2j*pi*c*n0/N) * X_fo[(k + ifo) mod N].  So while warp 0 runs the IFO search
        // (first bin of |fft(y3(Nfft+1:2*Nfft))| above 0.77; the window's constant phase exp(-2j*pi*fo) does not change
        // magnitudes and is skipped), warps 1..7 already transform symbols 0..6 with the fo-only table -- unpruned, since
        // the shift is not known yet -- and pick their bins once ifo is published.
        int ifo = 0;
        const int n_first = p.freq_desync ? min(NW - 1, p.S) : 0;
        if (p.freq_desync) {
            for (int i = tid; i < N; i += T4_THREADS) wtab[i] = rot_from_cycles(fo * (double)i / N);
            __syncthreads();
            float2 v[32];
            const int s1 = warp - 1;
            if (warp == 0) {
                load_window(r, (int64_t)N, tg, tshift, v);
#pragma unroll
                for (int n1 = 0; n1 < 32; ++n1) v[n1] = cmul(v[n1], wtab[32 * n1 + lane]);
                pass_a(v);
                fft32<32>(v);
                int first = 0x7fffffff;
#pragma unroll
                for (int k2 = 31; k2 >= 0; --k2) {
                    const double re = v[k2].x, im = v[k2].y;
                    if (sqrt(re * re + im * im) > 0.77) first = lane + 32 * k2;
                }
                first = warp_min(first);
                if (lane == 0) ifo_s = (first == 0x7fffffff) ? -1 : first;
            } else if (s1 < n_first) {
                load_window(r, (int64_t)s1 * SL + p.Tg, tg, tshift, v);
#pragma unroll
                for (int n1 = 0; n1 < 32; ++n1) v[n1] = cmul(v[n1], wtab[32 * n1 + lane]);
                pass_a(v);
                fft32<32>(v);
#pragma unroll
                for (int k2 = 0; k2 < 32; ++k2) E[lane + 32 * k2] = v[k2];      // whole spectrum, natural order, in the warp's tile
            }
        }
        if (p.freq_desync) {
            __syncthreads();
            ifo = ifo_s;
            const int s1 = warp - 1;
            if (warp > 0 && s1 < n_first) {
                const double c1 = fo + (ifo > 0 ? ifo : 0);
                const float2 rs = rot_from_cycles(c1 * (double)((int64_t)s1 * SL + p.Tg) / N);
                const int sh = ifo > 0 ? ifo : 0;
                for (int k = lane; k < p.Nc; k += 32) Ysc[(int64_t)s1 * p.Nc + k] = cmul(E[(k + sh) & (N - 1)], rs);
                for (int q = lane; q < p.Np; q += 32) Yp[s1 * p.Np + q] = cmul(E[(p.pil0[q] + sh) & (N - 1)], rs);
                __syncwarp();
            }
        }
        if (tid == 0 && ifo_out) ifo_out[b] = ifo;
        const double c = fo + (ifo > 0 ? ifo : 0);   // total derotation in cycles per Nfft samples
        if (tid == 0) next_sym = n_first;             // published by the barrier(s) below
        if (p.freq_desync) {
            __syncthreads();                          // every warp is done with the fo-only table
            if (ifo > 0) for (int i = tid; i < N; i += T4_THREADS) wtab[i] = rot_from_cycles(c * (double)i / N);
            for (int s = tid; s < p.S; s += T4_THREADS) rot_s[s] = rot_from_cycles(c * (double)((int64_t)s * SL + p.Tg) / N);
        }
        __syncthreads();
        // ---- OFDM_demodulator, one warp per symbol; park the useful bins (rotated), keep the pilots.  Symbols are handed
        // out through a shared counter: the warps did unequal work in the first round (IFO search / unpruned transforms).
        for (;;) {
            int s = 0;
            if (lane == 0) s = atomicAdd(&next_sym, 1);
            s = __shfl_sync(0xffffffffu, s, 0);
            if (s >= p.S) break;
            float2 v[32];
            load_window(r, (int64_t)s * SL + p.Tg, tg, tshift, v);
            if (p.freq_desync) {
#pragma unroll
                for (int n1 = 0; n1 < 32; ++n1) v[n1] = cmul(v[n1], wtab[32 * n1 + lane]);
            }
            pass_a(v);
            fft32<K2N>(v);
            const float2 rs = p.freq_desync ? rot_s[s] : make_float2(1.f, 0.f);
#pragma unroll
            for (int k2 = 0; k2 < K2N; ++k2) {
                const int k = lane + 32 * k2;
                const float2 y = p.freq_desync ? cmul(v[k2], rs) : v[k2];
                E[k] = y;                                                  // natural order, for the pilot gather below
                if (k < p.Nc) Ysc[(int64_t)s * p.Nc + k] = y;
            }
            __syncwarp();
            for (int q = lane; q < p.Np; q += 32) Yp[s * p.Np + q] = E[p.pil0[q]];
            __syncwarp();
        }
        __syncthreads();
        // ---- fine_sync estimators (`Task 4/fine_sync.m:25-35,47-52`), in double
        double tau = 0.0, phase = 0.0;
        if (p.time_desync || p.freq_desync) {
            const double deltak = (double)(p.pil0[1] - p.pil0[0]);
            // The pilots are FP32 DFT outputs: the products are formed in double, the angle itself in FP32 (its
            // argument carries no more than FP32 accuracy), sums and thresholds in double as in the reference.
            auto q_at = [&](int i) -> double2 { return cmulc(p.pilots_d[i], to_d(Yp[i])); };   // tx * conj(rx), flat column-major index
            auto tau_at = [&](int j) -> double { double2 d = cmulc(q_at(j + 1), q_at(j)); return (double)atan2f((float)d.y, (float)d.x) / (2.0 * CUDART_PI * deltak); };
            const int n = M - 1;
            for (int j = tid; j < n; j += T4_THREADS) taus[j] = tau_at(j);                  // taus(j+1) of the reference (:25-30)
            __syncthreads();
            // mask = [false, abs(diffs)<1e-3 & abs(diffs)~=0]; taus_result = taus(mask); mean(taus_result(Np+1:end))  (:32-35)
            const int CH = (n + T4_THREADS - 1) / T4_THREADS;
            const int lo = min(tid * CH, n), hi = min(lo + CH, n);
            int cmask = 0;
            for (int j = max(lo, 1); j < hi; ++j) { double d = fabs(taus[j] - taus[j - 1]); cmask += (d < 1e-3 && d != 0.0); }
            int rank = block_exclusive_scan(cmask, red_i);      // survivors before this thread's chunk
            double sum = 0; int kept = 0;
            for (int j = max(lo, 1); j < hi; ++j) {
                double d = fabs(taus[j] - taus[j - 1]);
                if (d < 1e-3 && d != 0.0) { if (rank >= p.Np) { sum += taus[j]; ++kept; } ++rank; }
            }
            sum = block_sum(sum, red);
            double nk = block_sum((double)kept, red);
            tau = sum / nk;
            // exp(+2j*pi*tau*k) at the pilot carriers, once per carrier (`fine_sync.m:38-44`); dk is free until the spline
            double2* prot = (double2*)taus;                                                 // taus is dead from here on
            __syncthreads();
            for (int q = tid; q < p.Np; q += T4_THREADS) {
                double sn = 0.0, cs = 1.0;
                if (p.time_desync) sincospi(2.0 * tau * (double)p.pil0[q], &sn, &cs);
                prot[q] = make_double2(cs, sn);
            }
            __syncthreads();
            double ps = 0; int pn = 0;
            for (int i = tid; i < M; i += T4_THREADS) {
                const int pq = i % p.Np;
                double2 rxv = to_d(Yp[i]);
                if (p.time_desync) rxv = cmul(rxv, prot[pq]);
                double2 qq = cmulc(p.pilots_d[i], rxv);
                double a = (double)atan2f((float)qq.y, (float)qq.x);
                if (fabs(a) > 1e-3) { ps += a; ++pn; }
            }
            ps = block_sum(ps, red);
            double pk = block_sum((double)pn, red);
            phase = ps / pk;
            if (tid == 0) { if (tau_out) tau_out[b] = tau; if (phase_out) phase_out[b] = phase; }
        }
        // ---- per-carrier correction factor exp(j*(2*pi*tau*k*[time] + phase*[freq])) (`fine_sync.m:38-58`)
        for (int k = tid; k < p.Nc; k += T4_THREADS) {
            double sn = 0.0, cs = 1.0;
            if (p.time_desync || p.freq_desync) {
                double ang = (p.time_desync ? 2.0 * tau * (double)k : 0.0);     // in units of pi
                double s1, c1, s2 = 0.0, c2 = 1.0;
                sincospi(ang, &s1, &c1);
                if (p.freq_desync) sincos(phase, &s2, &c2);
                cs = c1 * c2 - s1 * s2; sn = s1 * c2 + c1 * s2;
            }
            G[k] = make_float2((float)cs, (float)sn);
        }
        __syncthreads();
        // ---- estimate_channel on the corrected grid + equalize_signal (`estimate_channel.m:4-8`)
        if (p.mp_desync) {
            // mean over the symbols of rx_pilot * cf / tx_pilot (`estimate_channel.m:4-6`): one warp per pilot, lanes over the
            // symbols, summed in the reference's order only up to FP32 reassociation
            for (int q = warp; q < p.Np; q += NW) {
                float sr = 0.f, si = 0.f;
                const float2 g = G[p.pil0[q]];
                for (int s = lane; s < p.S; s += 32) { const float2 v = cdiv(cmul(Yp[s * p.Np + q], g), p.pilots[(int64_t)s * p.Np + q]); sr += v.x; si += v.y; }
                sr = warp_sum(sr); si = warp_sum(si);
                if (lane == 0) yk[q] = make_float2(sr / (float)p.S, si / (float)p.S);
            }
            __syncthreads();
            float2* Hrow = Hout ? Hout + b * p.Nc : nullptr;
            plan_apply_fn<float>(plan, yk, dk, [&](int k, float2 h) {
                if (Hrow) Hrow[k] = h;
                G[k] = cdiv(G[k], h);            // equalised = Y * cf / H
            });
            __syncthreads();
        }
        // ---- get_payload + demapping for the whole stream (decisions alias the tile/taus region, free by now)
        int errs = 0, nears = 0;
        uint8_t* dec = (uint8_t*)smem_raw;             // [S][Nd] codes = the stream's symbol order
        __syncthreads();
        for (int dr = tid; dr < p.Nd; dr += T4_THREADS) {
            const int cidx = p.data0[dr];
            const bool in = cidx < p.Nc;
            const float2 g = in ? G[cidx] : make_float2(0.f, 0.f);
            const float2* Yc = Ysc + (in ? cidx : 0);
            for (int s0 = 0; s0 < p.S; s0 += 10) {
                float2 y[10];
#pragma unroll
                for (int u = 0; u < 10; ++u) y[u] = (s0 + u < p.S) ? Yc[(int64_t)(s0 + u) * p.Nc] : make_float2(0.f, 0.f);
#pragma unroll
                for (int u = 0; u < 10; ++u)
                    if (s0 + u < p.S) {
                        const float2 e = in ? cmul(y[u], g) : make_float2(0.f, 0.f);
                        float margin = 1.f;
                        uint32_t code;
                        if (QAM16) code = demap16_nib<NEAR>(e.x, e.y, fx.two_a, &margin);
                        else code = (uint32_t)nearest_idx(con, e.x, e.y, &margin);
                        if (NEAR && margin < near_eps) ++nears;
                        dec[(s0 + u) * p.Nd + dr] = (uint8_t)code;
                    }
            }
        }
        __syncthreads();
        // ---- DeScrambler + BER
        if (QAM16 && (stream_bits & 31) == 0 && p.frame_bits >= 64) {
            // Word-aligned streams: raw stream word w = eight ready-made nibbles dec[8w .. 8w+7] (one 8-byte load); the
            // descrambler out[i] = raw[i] ^ raw[i-13] ^ raw[i-14] runs on a 64-bit window (previous word : this word).
            // Frames need not be word aligned (Task 4: 6,640 bits): where a frame starts at offset t inside the window the bits
            // below it are replaced by the initial register's history (`DeScrambler.m:8-13` with the per-frame reset of
            // `Main_model_Task_4.m:350-364`), and the word's bits before the boundary keep the previous frame's history.
            const int words = (int)(stream_bits >> 5);
            auto raw_word = [&](int w) -> uint32_t {
                const uint2 by = *reinterpret_cast<const uint2*>(dec + 8 * w);
                uint32_t lo = by.x | (by.x >> 4); lo = (lo & 0xFFu) | ((lo >> 8) & 0xFF00u);
                uint32_t hi = by.y | (by.y >> 4); hi = (hi & 0xFFu) | ((hi >> 8) & 0xFF00u);
                return lo | (hi << 16);
            };
            const uint32_t* tb = txbits ? txbits + b * words : nullptr;
            uint32_t* ob = outbits ? outbits + b * words : nullptr;
            for (int w = tid; w < words; w += T4_THREADS) {
                const uint32_t R = raw_word(w);
                uint32_t o = R;
                if (p.scramble) {                                   // descramble_word written out: the call reschedules this kernel
                    const uint32_t P = w ? raw_word(w - 1) : 0u;
                    const unsigned long long X = ((unsigned long long)R << 32) | P;
                    o = (uint32_t)((X ^ (X << 13) ^ (X << 14)) >> 32);
                    const int fl = (32 * w + 31) / p.frame_bits;            // frame of the word's last bit
                    const int t = fl * p.frame_bits - 32 * w;               // its start relative to this word: (-frame_bits, 31]
                    if (t > -14) {
                        const int sh = 32 + t;                              // window position of the frame's first bit, 19..63
                        const unsigned long long keep = ~0ull << sh;
                        const unsigned long long hist = sh >= 32 ? ((unsigned long long)p.prev0 << (sh - 32)) : ((unsigned long long)p.prev0 >> (32 - sh));
                        const unsigned long long Xf = (X & keep) | (hist & ~keep);
                        const uint32_t of = (uint32_t)((Xf ^ (Xf << 13) ^ (Xf << 14)) >> 32);
                        const uint32_t before = t > 0 ? ((1u << t) - 1u) : 0u;   // bits of this word that still belong to the previous frame
                        o = (o & before) | (of & ~before);
                    }
                }
                if (tb) errs += __popc(o ^ tb[w]);
                if (ob) ob[w] = o;
            }
        } else {
            // generic constellations / unaligned streams: frame by frame, a thread packs word wd and its predecessor itself
            const int fpb = p.SpF * p.Nd;              // decisions per frame
            auto packed = [&](const uint8_t* fr, int wd) -> uint32_t {
                uint32_t word = 0;
                if (QAM16) {                           // eight ready-made nibbles, one per byte (frames need not be 8-aligned in `dec`)
#pragma unroll
                    for (int j = 0; j < 8; ++j) { const int q = 8 * wd + j; if (q < fpb) word |= (uint32_t)fr[q] << (4 * j); }
                } else {
                    const int b0 = 32 * wd, b1 = min(b0 + 32, p.frame_bits);
                    for (int q = b0 / p.bps; q * p.bps < b1; ++q) {
                        int idx = fr[q];
                        for (int i = 0; i < p.bps; ++i) {
                            int pos = q * p.bps + i;
                            if (pos >= b0 && pos < b1 && ((idx >> (p.bps - 1 - i)) & 1)) word |= 1u << (pos - b0);
                        }
                    }
                }
                return word;
            };
            for (int item = tid; item < p.frames * fw; item += T4_THREADS) {
                const int f = item / fw, wd = item - f * fw;
                const uint8_t* fr = dec + (size_t)f * fpb;
                const uint32_t cw = packed(fr, wd);
                uint32_t o = cw;
                if (p.scramble) {
                    const uint32_t prev = wd ? packed(fr, wd - 1) : p.prev0;
                    o = cw ^ ((cw << 13) | (prev >> 19)) ^ ((cw << 14) | (prev >> 18));
                }
                const int n = min(32, p.frame_bits - 32 * wd);
                if (n < 32) o &= (1u << n) - 1u;
                const int64_t base = b * stream_bits + (int64_t)f * p.frame_bits;
                if (txbits) errs += __popc(o ^ bits_get32(txbits, base + 32 * (int64_t)wd, min(total_bits, base + p.frame_bits)));
                if (outbits) bits_put(outbits, base + 32 * (int64_t)wd, n, o);
            }
        }
        errs = block_sum(errs, red_i);
        nears = block_sum(nears, red_i);
        if (tid == 0 && counts) {
            if (errs) atomicAdd(&counts[0], (unsigned long long)errs);
            atomicAdd(&counts[1], (unsigned long long)stream_bits);
            if (nears) atomicAdd(&counts[2], (unsigned long long)nears);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------
// Split form of the fast path (large batches): the same arithmetic as rx_t4_fast_kernel in three kernels, so that each
// part runs at its own occupancy instead of sharing one 128-register, two-CTA-per-SM persistent kernel:
//   t4_ifo_kernel    one warp per stream: remove_IFO's search (`remove_IFO.m:5-8`)
//   t4_sym_kernel    one CTA per (stream, eight symbols): derotation + 1024-point DFT per warp, no block barrier after the
//                    rotation table; writes the N_carrier kept bins and the pilots of every symbol
//   t4_post_kernel   one CTA per stream, few registers: fine_sync estimators, channel estimate, decisions, DeScrambler, BER
// The kept bins travel through global memory (N_carrier x S complex per stream) instead of a per-CTA L2 parking area.
__device__ __forceinline__ void t4_load_window(const float2* __restrict__ r, int64_t L, int SL, int64_t n0, int tg, bool tshift, int lane, float2* v) {
    constexpr int N = 1024;
    const int64_t m0 = tshift ? n0 - SL + tg : n0;          // sample n of the corrected stream is r[n - SL + tg] for n >= SL, else 0 (`add_STO.m:5-9`)
    const bool all_in = (m0 >= 0 && m0 + N <= L && (!tshift || n0 >= SL));
    if (all_in) {
        const float2* q = r + m0 + lane;
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) v[n1] = ldg_stream(q + 32 * n1);
    } else {
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) {
            const int64_t m = m0 + 32 * n1 + lane;
            const bool ok = m >= 0 && m < L && (!tshift || n0 + 32 * n1 + lane >= SL);
            v[n1] = ok ? ldg_stream(r + m) : make_float2(0.f, 0.f);
        }
    }
}
__device__ __forceinline__ void t4_pass_a(float2* v, float2* E, const float2* __restrict__ tw_t, int lane) {   // DFT over n1, twiddle, transpose
    fft32<32>(v);
#pragma unroll
    for (int k1 = 0; k1 < 32; ++k1) {
        float2 x = v[k1];
        if (k1) x = cmul(x, __ldg(tw_t + 32 * k1 + lane));
        E[k1 * T4F_EROW + lane] = x;
    }
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; ++n2) v[n2] = E[lane * T4F_EROW + n2];
    __syncwarp();
}

__global__ void __launch_bounds__(T4_THREADS) t4_ifo_kernel(T4FastExtra fx, const float2* __restrict__ rx, int64_t B, int64_t L, int Tg, int time_desync,
                                                            const int32_t* __restrict__ tg_pos, const double* __restrict__ freq_off,
                                                            int32_t* __restrict__ ifo_out) {
    constexpr int N = 1024;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t b = (int64_t)blockIdx.x * (T4_THREADS / 32) + warp;
    if (b >= B) return;
    float2* E = (float2*)smem_raw + warp * 32 * T4F_EROW;
    const double fo = freq_off[b];
    float2 v[32];
    t4_load_window(rx + b * L, L, N + Tg, (int64_t)N, time_desync ? tg_pos[b] : 0, time_desync != 0, lane, v);
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) v[n1] = cmul(v[n1], rot_from_cycles(fo * (double)(32 * n1 + lane) / N));   // the window's constant phase does not change magnitudes
    t4_pass_a(v, E, fx.tw_t, lane);
    fft32<32>(v);
    int first = 0x7fffffff;
#pragma unroll
    for (int k2 = 31; k2 >= 0; --k2) {
        const double re = v[k2].x, im = v[k2].y;
        if (sqrt(re * re + im * im) > 0.77) first = lane + 32 * k2;
    }
    first = warp_min(first);
    if (lane == 0) ifo_out[b] = (first == 0x7fffffff) ? -1 : first;
}

template <int K2N>
__global__ void __launch_bounds__(T4_THREADS, 2) t4_sym_kernel(T4Params p, T4FastExtra fx, const float2* __restrict__ rx, int64_t B, int64_t L, int groups,
                                                               const int32_t* __restrict__ tg_pos, const double* __restrict__ freq_off,
                                                               const int32_t* __restrict__ ifo_in, float2* __restrict__ Yd_all, float2* __restrict__ Yp_all) {
    constexpr int N = 1024;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NW = T4_THREADS / 32;
    float2* tiles = (float2*)smem_raw;
    float2* wtab = tiles + NW * 32 * T4F_EROW;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b = blockIdx.x / groups;
    const int g = (int)(blockIdx.x - b * groups);
    const int SL = N + p.Tg;
    const int tg = p.time_desync ? tg_pos[b] : 0;
    const int ifo = p.freq_desync ? ifo_in[b] : 0;
    const double c = (p.freq_desync ? freq_off[b] : 0.0) + (ifo > 0 ? ifo : 0);     // total derotation in cycles per Nfft samples
    if (p.freq_desync) {
        for (int i = tid; i < N; i += T4_THREADS) wtab[i] = rot_from_cycles(c * (double)i / N);
        __syncthreads();
    }
    const int s = NW * g + warp;
    if (s >= p.S) return;
    float2* E = tiles + warp * 32 * T4F_EROW;
    float2 v[32];
    t4_load_window(rx + b * L, L, SL, (int64_t)s * SL + p.Tg, tg, p.time_desync != 0, lane, v);
    if (p.freq_desync) {
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) v[n1] = cmul(v[n1], wtab[32 * n1 + lane]);
    }
    t4_pass_a(v, E, fx.tw_t, lane);
    fft32<K2N>(v);
    const float2 rs = p.freq_desync ? rot_from_cycles(c * (double)((int64_t)s * SL + p.Tg) / N) : make_float2(1.f, 0.f);
#pragma unroll
    for (int k2 = 0; k2 < K2N; ++k2) {
        const float2 y = p.freq_desync ? cmul(v[k2], rs) : v[k2];
        E[lane + 32 * k2] = (lane + 32 * k2 < p.Nc) ? y : make_float2(0.f, 0.f);      // natural order, for the two gathers below (`get_payload.m`, pilots)
    }
    __syncwarp();
    // data carriers in payload order, pilots in pilot order: the post kernel reads both linearly
    float2* Yo = Yd_all + ((int64_t)b * p.S + s) * p.Nd;
    if ((p.Nd & 1) == 0) {
        const int2* d2 = reinterpret_cast<const int2*>(p.data0);
        for (int h = lane; 2 * h < p.Nd; h += 32) {
            const int2 c = __ldg(d2 + h);
            const float2 y0 = c.x < 32 * K2N ? E[c.x] : make_float2(0.f, 0.f), y1 = c.y < 32 * K2N ? E[c.y] : make_float2(0.f, 0.f);
            reinterpret_cast<float4*>(Yo)[h] = make_float4(y0.x, y0.y, y1.x, y1.y);
        }
    } else {
        for (int dr = lane; dr < p.Nd; dr += 32) { const int c = p.data0[dr]; Yo[dr] = c < 32 * K2N ? E[c] : make_float2(0.f, 0.f); }
    }
    float2* Po = Yp_all + ((int64_t)b * p.S + s) * p.Np;
    for (int q = lane; q < p.Np; q += 32) Po[q] = E[p.pil0[q]];
}

// Statistics of the sweep variant (t4_post_kernel<Q, false, true>, ofdm_sweep_sync): what the stream's receiver reports besides its bits.
struct T4Stats {
    const double2* Htrue;      // true response H(1:N_carrier), double
    double* rec;               // 9 fields x rec_stride doubles; this launch's stream b at rec[f * rec_stride + b]
    int64_t rec_stride;
    const int32_t* tg;         // TgPosition, FreqOffset, IFO, guard-detector failure flag (NULL: detector not run), true STO / CFO
    const double* fo;
    const int32_t* ifo;
    const int32_t* fail;
    const int32_t* nsto;
    const double* cfo;
    float a_in, a_out;         // 16QAM: |levels| of the inner and outer points per axis
};
// 16QAM point nearest to e, per axis (the separable rule of demap16_nib), accumulated as `MER_func.m:7-25` does.  It is the
// point MER_func's abs() search returns except for exact ties on a decision boundary, where either point is equally near.
__device__ __forceinline__ void t4_mer16(float2 e, float two_a, float a_in, float a_out, double& s1, double& s2) {
    const float ix = copysignf(fabsf(e.x) < two_a ? a_in : a_out, e.x), iy = copysignf(fabsf(e.y) < two_a ? a_in : a_out, e.y);
    const double er = (double)ix - (double)e.x, ei = (double)iy - (double)e.y;
    s1 += (double)ix * ix + (double)iy * iy;
    s2 += er * er + ei * ei;
}

// STATS (ofdm_sweep_sync, NEAR false): the same chain and arithmetic without output bits, tau / phase, H or near-boundary
// count, and the same CTA also
//   * accumulates the channel-estimate error sum |H_est(k) - H(k)|^2 in double against st.Htrue while the spline emits H_est
//     (never stored), with mse_kernel's terms;
//   * accumulates the MER sums of `MER_func.m:7-25` while the data carriers are decided;
//   * reduces both with the fixed-order block_sum, writes the stream's record and adds {detector failure, IFO = -1} to the
//     point's row {errors, bits, detector failures, IFO misses} with integer atomics.
// st is the last parameter so that the other parameters keep their offsets; the kernels without STATS do not read it.
template <bool QAM16, bool NEAR, bool STATS>
__global__ void __launch_bounds__(T4_THREADS, 4) t4_post_kernel(T4Params p, T4FastExtra fx, PlanDev<float> plan, DevConst<float> con, int64_t B,
                                                                const float2* __restrict__ Yd_all, const float2* __restrict__ Yp_all,
                                                                const uint32_t* __restrict__ txbits, int64_t total_bits, uint32_t* __restrict__ outbits,
                                                                unsigned long long* __restrict__ counts, double* __restrict__ tau_out,
                                                                double* __restrict__ phase_out, float2* __restrict__ Hout, float near_eps, T4Stats st) {
    if constexpr (STATS) {                                       // switched-off outputs: their branches go at compile time
        outbits = nullptr; tau_out = nullptr; phase_out = nullptr; Hout = nullptr; near_eps = 0.f;
    }
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double red[32];
    __shared__ int red_i[32];
    const int tid = threadIdx.x, lane = tid & 31;
    const int M = p.Np * p.S;
    // layout: region A = [angles (float) | rotations | decisions / raw words] (aliased in time), Yp (later: partial sums, then Gd), G, yk, dk
    const size_t ang_bytes = sizeof(float) * (size_t)M, rot_bytes = sizeof(double2) * (size_t)p.Np, dec_bytes = (size_t)p.S * p.Nd;
    float* ang = (float*)smem_raw;
    float2* Yp = (float2*)(smem_raw + (max(max(ang_bytes, rot_bytes), max(dec_bytes, sizeof(float2) * (size_t)T4_THREADS)) + 15) / 16 * 16);
    float2* G = Yp + M;
    float2* yk = G + p.Nc;
    float2* dk = yk + plan.n_knots;
    const int fw = (p.frame_bits + 31) >> 5;
    const int64_t b = blockIdx.x;
    const float2* Yd = Yd_all + b * (int64_t)p.S * p.Nd;
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
    const int step_q = T4_THREADS % p.Np;                    // pilot index of item i = tid + T4_THREADS * j, advanced without a division
    {
        const float2* src = Yp_all + b * (int64_t)M;
        for (int i = tid; i < M; i += T4_THREADS) Yp[i] = src[i];
    }
    __syncthreads();
    // ---- fine_sync estimators (`Task 4/fine_sync.m:25-35,47-52`), products in double, angles in FP32 (as in the fused kernel)
    double tau = 0.0, phase = 0.0;
    if (p.time_desync || p.freq_desync) {
        const double inv_c = 1.0 / (2.0 * CUDART_PI * (double)(p.pil0[1] - p.pil0[0]));       // tau_j = angle_j / (2 pi deltak)
        auto q_at = [&](int i) -> double2 { return cmulc(p.pilots_d[i], to_d(Yp[i])); };
        const int n = M - 1;
        for (int j0 = 0; j0 < n; j0 += T4_THREADS) {          // angle of q_{j+1} conj(q_j): q_j once per thread, q_{j+1} from the next lane
            const int j = j0 + tid;
            double2 qa = make_double2(0.0, 0.0), qb;
            if (j < M) qa = q_at(j);
            qb.x = __shfl_down_sync(0xffffffffu, qa.x, 1);
            qb.y = __shfl_down_sync(0xffffffffu, qa.y, 1);
            if (lane == 31 && j + 1 < M) qb = q_at(j + 1);
            if (j < n) { const double2 d = cmulc(qb, qa); ang[j] = atan2f((float)d.y, (float)d.x); }
        }
        __syncthreads();
        const int CH = (n + T4_THREADS - 1) / T4_THREADS;
        const int lo = min(tid * CH, n), hi = min(lo + CH, n);
        int cmask = 0;
        for (int j = max(lo, 1); j < hi; ++j) { double d = fabs((double)ang[j] - (double)ang[j - 1]) * inv_c; cmask += (d < 1e-3 && d != 0.0); }   // the difference first: exactly zero for equal angles
        int rank = block_exclusive_scan(cmask, red_i);
        double sum = 0; int kept = 0;
        for (int j = max(lo, 1); j < hi; ++j) {
            const double tj = (double)ang[j] * inv_c, d = fabs((double)ang[j] - (double)ang[j - 1]) * inv_c;
            if (d < 1e-3 && d != 0.0) { if (rank >= p.Np) { sum += tj; ++kept; } ++rank; }
        }
        sum = block_sum(sum, red);
        double nk = block_sum((double)kept, red);
        tau = sum / nk;
        double2* prot = (double2*)smem_raw;
        __syncthreads();
        for (int q = tid; q < p.Np; q += T4_THREADS) {
            double sn = 0.0, cs = 1.0;
            if (p.time_desync) sincospi(2.0 * tau * (double)p.pil0[q], &sn, &cs);
            prot[q] = make_double2(cs, sn);
        }
        __syncthreads();
        double ps = 0; int pn = 0;
        for (int i = tid, pq = tid % p.Np; i < M; i += T4_THREADS) {
            double2 rxv = to_d(Yp[i]);
            if (p.time_desync) rxv = cmul(rxv, prot[pq]);
            double2 qq = cmulc(p.pilots_d[i], rxv);
            double a = (double)atan2f((float)qq.y, (float)qq.x);
            if (fabs(a) > 1e-3) { ps += a; ++pn; }
            pq += step_q; if (pq >= p.Np) pq -= p.Np;
        }
        ps = block_sum(ps, red);
        double pk = block_sum((double)pn, red);
        phase = ps / pk;
        if (tid == 0) { if (tau_out) tau_out[b] = tau; if (phase_out) phase_out[b] = phase; }
    }
    {
        double s2 = 0.0, c2 = 1.0;
        if (p.freq_desync) sincos(phase, &s2, &c2);
        for (int k = tid; k < p.Nc; k += T4_THREADS) {
            double sn = 0.0, cs = 1.0;
            if (p.time_desync || p.freq_desync) {
                double s1, c1;
                sincospi(p.time_desync ? 2.0 * tau * (double)k : 0.0, &s1, &c1);
                cs = c1 * c2 - s1 * s2; sn = s1 * c2 + c1 * s2;
            }
            G[k] = make_float2((float)cs, (float)sn);
        }
    }
    __syncthreads();
    double herr = 0.0, mer1 = 0.0, mer2 = 0.0;                   // STATS only
    if (p.mp_desync) {
        // symbol-averaged pilot LS values: PARTS threads per pilot (consecutive lanes = consecutive pilots: conflict-free shared
        // reads, coalesced pilot table), partial sums combined in a fixed order
        const int PARTS = min(min(T4_THREADS / p.Np, 4), p.S);
        float2* part = (float2*)smem_raw;
        if (tid < PARTS * p.Np) {
            const int pt = tid / p.Np, q = tid - pt * p.Np;
            const float2 g = G[p.pil0[q]];
            float sr = 0.f, si = 0.f;
            for (int s = pt; s < p.S; s += PARTS) { const float2 v = cdiv(cmul(Yp[s * p.Np + q], g), p.pilots[(int64_t)s * p.Np + q]); sr += v.x; si += v.y; }
            part[tid] = make_float2(sr, si);
        }
        __syncthreads();
        for (int q = tid; q < p.Np; q += T4_THREADS) {
            float sr = 0.f, si = 0.f;
            for (int pt = 0; pt < PARTS; ++pt) { sr += part[pt * p.Np + q].x; si += part[pt * p.Np + q].y; }
            yk[q] = make_float2(sr / (float)p.S, si / (float)p.S);
        }
        __syncthreads();
        float2* Hrow = Hout ? Hout + b * p.Nc : nullptr;
        plan_apply_fn<float>(plan, yk, dk, [&](int k, float2 h) {
            if (Hrow) Hrow[k] = h;
            if constexpr (STATS) {
                const double2 t = st.Htrue[k];                   // the terms of mse_kernel, in double
                const double dr = t.x - (double)h.x, di = t.y - (double)h.y;
                herr += dr * dr + di * di;
            }
            G[k] = cdiv(G[k], h);
        });
    }
    __syncthreads();
    float2* Gd = Yp;                                             // one-tap equaliser of the data carriers in payload order
    for (int dr = tid; dr < p.Nd; dr += T4_THREADS) { const int c = p.data0[dr]; Gd[dr] = c < p.Nc ? G[c] : make_float2(0.f, 0.f); }
    __syncthreads();
    int errs = 0, nears = 0;
    if (QAM16 && (stream_bits & 31) == 0 && p.frame_bits >= 64 && (p.Nd & 3) == 0) {
        // word-aligned 16QAM streams: one thread decides the eight consecutive payload symbols of a 32-bit word (64 contiguous
        // bytes of the compact data-carrier array); a group of four never straddles two OFDM symbols because Nd % 4 == 0
        const int words = (int)(stream_bits >> 5);
        uint32_t* rawW = (uint32_t*)smem_raw;
        const float4* Yv = reinterpret_cast<const float4*>(Yd);
        for (int w = tid; w < words; w += T4_THREADS) {
            float4 y[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) y[u] = __ldg(Yv + 4 * w + u);
            const int i0 = 8 * w;
            const int dr0 = i0 - (i0 / p.Nd) * p.Nd;
            const int dr1 = dr0 + 4 >= p.Nd ? 0 : dr0 + 4;
            float4 g[4];
            g[0] = *reinterpret_cast<const float4*>(Gd + dr0); g[1] = *reinterpret_cast<const float4*>(Gd + dr0 + 2);
            g[2] = *reinterpret_cast<const float4*>(Gd + dr1); g[3] = *reinterpret_cast<const float4*>(Gd + dr1 + 2);
            uint32_t R = 0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float2 e0 = cmul(make_float2(y[u].x, y[u].y), make_float2(g[u].x, g[u].y));
                const float2 e1 = cmul(make_float2(y[u].z, y[u].w), make_float2(g[u].z, g[u].w));
                float m0 = 1.f, m1 = 1.f;
                R |= demap16_nib<NEAR>(e0.x, e0.y, fx.two_a, &m0) << (8 * u);
                R |= demap16_nib<NEAR>(e1.x, e1.y, fx.two_a, &m1) << (8 * u + 4);
                if (NEAR) nears += (m0 < near_eps) + (m1 < near_eps);
                if constexpr (STATS) {
                    t4_mer16(e0, fx.two_a, st.a_in, st.a_out, mer1, mer2);
                    t4_mer16(e1, fx.two_a, st.a_in, st.a_out, mer1, mer2);
                }
            }
            rawW[w] = R;
        }
        __syncthreads();
        const uint32_t* tb = txbits ? txbits + b * words : nullptr;
        uint32_t* ob = outbits ? outbits + b * words : nullptr;
        for (int w = tid; w < words; w += T4_THREADS) {
            const uint32_t R = rawW[w];
            uint32_t o = R;
            if (p.scramble) {                                       // descramble_word written out: the call reschedules this kernel
                const uint32_t P = w ? rawW[w - 1] : 0u;
                const unsigned long long X = ((unsigned long long)R << 32) | P;
                o = (uint32_t)((X ^ (X << 13) ^ (X << 14)) >> 32);
                const int fl = (32 * w + 31) / p.frame_bits;
                const int t = fl * p.frame_bits - 32 * w;
                if (t > -14) {
                    const int sh = 32 + t;
                    const unsigned long long keep = ~0ull << sh;
                    const unsigned long long hist = sh >= 32 ? ((unsigned long long)p.prev0 << (sh - 32)) : ((unsigned long long)p.prev0 >> (32 - sh));
                    const unsigned long long Xf = (X & keep) | (hist & ~keep);
                    const uint32_t of = (uint32_t)((Xf ^ (Xf << 13) ^ (Xf << 14)) >> 32);
                    const uint32_t before = t > 0 ? ((1u << t) - 1u) : 0u;
                    o = (o & before) | (of & ~before);
                }
            }
            if (tb) errs += __popc(o ^ tb[w]);
            if (ob) ob[w] = o;
        }
    } else {
        uint8_t* dec = (uint8_t*)smem_raw;
        for (int dr = tid; dr < p.Nd; dr += T4_THREADS) {
            const float2 g = Gd[dr];
            const float2* Yc = Yd + dr;
            for (int s0 = 0; s0 < p.S; s0 += 10) {
                float2 y[10];
#pragma unroll
                for (int u = 0; u < 10; ++u) y[u] = (s0 + u < p.S) ? ldg_stream(Yc + (int64_t)(s0 + u) * p.Nd) : make_float2(0.f, 0.f);
#pragma unroll
                for (int u = 0; u < 10; ++u)
                    if (s0 + u < p.S) {
                        const float2 e = cmul(y[u], g);
                        float margin = 1.f;
                        uint32_t code;
                        if (QAM16) code = demap16_nib<NEAR>(e.x, e.y, fx.two_a, &margin);
                        else code = (uint32_t)nearest_idx(con, e.x, e.y, &margin);
                        if (NEAR && margin < near_eps) ++nears;
                        if constexpr (STATS) {
                            if (QAM16) t4_mer16(e, fx.two_a, st.a_in, st.a_out, mer1, mer2);
                            else {                               // `MER_func.m:7-25` as mer_kernel: the decided (nearest) point
                                const double ir = con.re[code], ii = con.im[code], er = ir - (double)e.x, ei = ii - (double)e.y;
                                mer1 += ir * ir + ii * ii;
                                mer2 += er * er + ei * ei;
                            }
                        }
                        dec[(s0 + u) * p.Nd + dr] = (uint8_t)code;
                    }
            }
        }
        __syncthreads();
        const int fpb = p.SpF * p.Nd;
        auto packed = [&](const uint8_t* fr, int wd) -> uint32_t {
            uint32_t word = 0;
            if (QAM16) {
#pragma unroll
                for (int j = 0; j < 8; ++j) { const int q = 8 * wd + j; if (q < fpb) word |= (uint32_t)fr[q] << (4 * j); }
            } else {
                const int b0 = 32 * wd, b1 = min(b0 + 32, p.frame_bits);
                for (int q = b0 / p.bps; q * p.bps < b1; ++q) {
                    int idx = fr[q];
                    for (int i = 0; i < p.bps; ++i) {
                        int pos = q * p.bps + i;
                        if (pos >= b0 && pos < b1 && ((idx >> (p.bps - 1 - i)) & 1)) word |= 1u << (pos - b0);
                    }
                }
            }
            return word;
        };
        for (int item = tid; item < p.frames * fw; item += T4_THREADS) {
            const int f = item / fw, wd = item - f * fw;
            const uint8_t* fr = dec + (size_t)f * fpb;
            const uint32_t cw = packed(fr, wd);
            uint32_t o = cw;
            if (p.scramble) {
                const uint32_t prev = wd ? packed(fr, wd - 1) : p.prev0;
                o = cw ^ ((cw << 13) | (prev >> 19)) ^ ((cw << 14) | (prev >> 18));
            }
            const int n = min(32, p.frame_bits - 32 * wd);
            if (n < 32) o &= (1u << n) - 1u;
            const int64_t base = b * stream_bits + (int64_t)f * p.frame_bits;
            if (txbits) errs += __popc(o ^ bits_get32(txbits, base + 32 * (int64_t)wd, min(total_bits, base + p.frame_bits)));
            if (outbits) bits_put(outbits, base + 32 * (int64_t)wd, n, o);
        }
    }
    errs = block_sum(errs, red_i);
    nears = block_sum(nears, red_i);
    if (tid == 0 && counts) {
        if (errs) atomicAdd(&counts[0], (unsigned long long)errs);
        atomicAdd(&counts[1], (unsigned long long)stream_bits);
        if (nears) atomicAdd(&counts[2], (unsigned long long)nears);
    }
    if constexpr (STATS) {
        herr = block_sum(herr, red);                              // fixed-order block reductions
        mer1 = block_sum(mer1, red);
        mer2 = block_sum(mer2, red);
        if (tid == 0) {
            const int ifo = p.freq_desync ? st.ifo[b] : 0;
            const int fail = st.fail ? st.fail[b] : 0;
            double* r = st.rec + b;
            const int64_t sd = st.rec_stride;
            r[0] = p.time_desync ? (double)st.tg[b] : 0.0;
            r[sd] = p.freq_desync ? st.fo[b] : 0.0;
            r[2 * sd] = (double)ifo;
            r[3 * sd] = tau;
            r[4 * sd] = phase;
            r[5 * sd] = p.mp_desync ? herr / (double)p.Nc : CUDART_NAN;
            r[6 * sd] = 10.0 * log10(mer1 / mer2);
            r[7 * sd] = (double)st.nsto[b];
            r[8 * sd] = st.cfo[b];
            if (fail) atomicAdd(&counts[2], 1ull);                    // row {errors, bits, detector failures, IFO misses}
            if (ifo < 0) atomicAdd(&counts[3], 1ull);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// TX side of the Task-4 shape (Nfft = 1024), same structure as t4_sym_kernel run backwards: one CTA per stream scrambles all
// of its frames at once in shared memory (log-depth GF(2) products, as tx_chain_kernel), then ONE WARP builds and transforms
// a symbol: lane m2 forms the (conjugated) carriers 32 m1 + m2 straight from the frame's bit array, DFT over m1 in
// registers, twiddle, 32 x 33 transpose, DFT over m2; lane j1 then holds the samples n = j1 + 32 j2, every store is a
// 256-byte row, rows j2 >= (1024 - Tg) / 32 are written a second time as the cyclic prefix (`OFDM_modulator.m:5-9`).
// ifft(X) = conj(fft(conj(X))) / N.  Replaces scrambler / mapping / OFDM_map_carriers / OFDM_modulator for this shape.
struct Tx1024Params {
    int Tg, Nc, S, SpF, Nd, Np, bps, scramble, frame_bits, frames, m1n;
    uint32_t prev0;
    const int32_t* slot;       // 1024: data rank / -1-pilot / SLOT_ZERO
    const float2* pilots;      // Np x S column-major
    const float2* tw_t;
};
#define T4_SLOT_ZERO (-2147483647 - 1)
__device__ __forceinline__ uint32_t t4_sm_get32(const uint32_t* w, int pos, int nwords) {     // 32 bits from bit `pos` of a frame array; outside reads 0
    if (pos < 0) return pos <= -32 ? 0u : w[0] << (-pos);
    const int wi = pos >> 5, sh = pos & 31;
    const uint32_t lo = wi < nwords ? w[wi] : 0u;
    const uint32_t hi = (sh && wi + 1 < nwords) ? w[wi + 1] : 0u;
    return __funnelshift_r(lo, hi, sh);
}
__global__ void __launch_bounds__(T4_THREADS, 2) tx1024_kernel(Tx1024Params p, DevConst<float> con, const uint32_t* __restrict__ bits, int64_t total_bits,
                                                               float2* __restrict__ out, double* __restrict__ power_part) {
    constexpr int N = 1024;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NW = T4_THREADS / 32;
    float2* tiles = (float2*)smem_raw;
    const int fw = (p.frame_bits + 31) >> 5;
    const int fwp = fw + 1;                                    // one zero word after every frame: unconditional two-word bit fetches
    uint32_t* s0 = (uint32_t*)(tiles + NW * 32 * T4F_EROW);
    uint32_t* s1 = s0 + p.frames * fwp;
    __shared__ float2 cs[16];                                  // conjugated constellation
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b = blockIdx.x;
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
    if (tid < 16) cs[tid] = make_float2(con.re[tid], -con.im[tid]);
    for (int i = tid; i < p.frames * fwp; i += T4_THREADS) {
        const int f = i / fwp, w = i - f * fwp;
        const int64_t base = b * stream_bits + (int64_t)f * p.frame_bits;
        uint32_t v = w < fw ? bits_get32(bits, base + 32 * (int64_t)w, min(total_bits, base + p.frame_bits)) : 0u;
        if (w == 0 && p.scramble) v ^= (p.prev0 >> 19) ^ (p.prev0 >> 18);     // fold the register pre-history into the input
        s0[i] = v;
        s1[i] = 0u;
    }
    __syncthreads();
    uint32_t* cur = s0; uint32_t* nxt = s1;
    if (p.scramble) {
        // s = in' * prod_j (1 + x^(13*2^j) + x^(14*2^j)) over GF(2), 13*2^j < frame_bits, every frame of the stream in the same round
        for (int sh13 = 13, sh14 = 14; sh13 < p.frame_bits; sh13 <<= 1, sh14 <<= 1) {
            for (int i = tid; i < p.frames * fw; i += T4_THREADS) {
                const int f = i / fw, w = i - f * fw;
                const uint32_t* cf = cur + f * fwp;
                nxt[f * fwp + w] = cf[w] ^ t4_sm_get32(cf, 32 * w - sh13, fw) ^ t4_sm_get32(cf, 32 * w - sh14, fw);
            }
            __syncthreads();
            uint32_t* t = cur; cur = nxt; nxt = t;
        }
    }
    float2* E = tiles + warp * 32 * T4F_EROW;
    const float inv_n = 1.f / N;
    // roles of this lane's carriers 32 m1 + lane, once for all symbols (only m1 < m1n <= 32 can be occupied)
    int sl[32];
#pragma unroll
    for (int m1 = 0; m1 < 32; ++m1) sl[m1] = m1 < p.m1n ? __ldg(p.slot + 32 * m1 + lane) : T4_SLOT_ZERO;
    for (int s = warp; s < p.S; s += NW) {
        const int f = s / p.SpF, sf = s - f * p.SpF;
        const uint32_t* cf = cur + f * fwp;
        const float2* prow = p.pilots + (int64_t)s * p.Np;
        float2 v[32];
        // all fetches first (independent), the selects after
#pragma unroll
        for (int m1 = 0; m1 < 32; ++m1) {
            float2 x = make_float2(0.f, 0.f);
            if (m1 < p.m1n) {
                const int r = sl[m1];
                if (r >= 0) {
                    const int pos = (sf * p.Nd + r) * p.bps;
                    const uint32_t g = __funnelshift_r(cf[pos >> 5], cf[(pos >> 5) + 1], pos & 31);
                    x = cs[__brev(g) >> (32 - p.bps)];                 // the symbol's bits, first bit most significant (`mapping.m`)
                } else if (r != T4_SLOT_ZERO) {
                    const float2 pv = __ldg(prow + (-1 - r));
                    x = make_float2(pv.x, -pv.y);
                }
            }
            v[m1] = x;
        }
        t4_pass_a(v, E, p.tw_t, lane);
        fft32<32>(v);
        float2* dst = out + (b * p.S + s) * (int64_t)(N + p.Tg);
        const int cp0 = N - p.Tg;
        float psym = 0.f;                                      // this lane's share of sum |x|^2 over the symbol, cyclic prefix included
#pragma unroll
        for (int j2 = 0; j2 < 32; ++j2) {
            const int n = lane + 32 * j2;
            const float2 y = make_float2(v[j2].x * inv_n, -v[j2].y * inv_n);
            dst[p.Tg + n] = y;
            if (n >= cp0) dst[n - cp0] = y;
            const float e = y.x * y.x + y.y * y.y;
            psym += n >= cp0 ? e + e : e;
        }
        if (power_part) {                                      // `Noise.m:3`: one partial per symbol, added up in symbol order afterwards (deterministic)
            const double tot = warp_sum((double)psym);
            if (lane == 0) power_part[b * p.S + s] = tot;
        }
    }
}

const void* t4_twiddle_blob(ofdm_ctx* ctx) {          // [k1][n2] = W1024^{n2 k1}
    std::vector<float> twt(2 * 1024);
    for (int k1 = 0; k1 < 32; ++k1)
        for (int n2 = 0; n2 < 32; ++n2) {
            const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double)((n2 * k1) & 1023) / 1024.0L;
            twt[2 * (32 * k1 + n2)] = (float)cosl(a); twt[2 * (32 * k1 + n2) + 1] = (float)sinl(a);
        }
    return ctx_blob(ctx, twt.data(), sizeof(float) * twt.size());
}

// TX chain fast path for Nfft = 1024 (FP32, every carrier inside N_carrier).  Sets *handled when it ran.
int ofdm_power_finish(ofdm_ctx* ctx, const double* partial, int64_t B, int nb, double* power_sum);      // channel.cu
int ofdm_tx1024_fast(ofdm_ctx* ctx, const ofdm_link_params* lp, const uint32_t* bits, int64_t B, void* time, double* power, bool* handled) {
    *handled = false;
    if (ctx->precision != OFDM_PREC_F32 || !lp || lp->Nfft != 1024 || getenv("OFDM_B200_NO_FAST")) return OFDM_OK;
    if (lp->S <= 0 || lp->SpF <= 0 || lp->S % lp->SpF || lp->Nd < 1 || lp->Np < 1 || lp->Tg < 0 || lp->Tg > 1024 || lp->N_carrier < 2 || lp->N_carrier > 1024) return OFDM_OK;
    ConstTable ct = host_constellation(lp->constellation);
    if (ct.bps <= 0 || (1 << ct.bps) > 16) return OFDM_OK;
    std::vector<int32_t> slot(1024, T4_SLOT_ZERO);
    for (int i = 0; i < lp->Nd; ++i) { const int c = lp->data_carriers_host[i]; if (c < 1 || c > lp->N_carrier) return OFDM_OK; slot[c - 1] = i; }
    for (int i = 0; i < lp->Np; ++i) { const int c = lp->pilot_carriers_host[i]; if (c < 1 || c > lp->N_carrier) return OFDM_OK; slot[c - 1] = -1 - i; }
    Tx1024Params p;
    p.Tg = lp->Tg; p.Nc = lp->N_carrier; p.S = lp->S; p.SpF = lp->SpF; p.Nd = lp->Nd; p.Np = lp->Np; p.bps = ct.bps; p.scramble = lp->scramble;
    p.frame_bits = lp->SpF * lp->Nd * ct.bps; p.frames = lp->S / lp->SpF; p.m1n = (lp->N_carrier + 31) / 32;
    p.prev0 = ofdm_reg_to_prev(lp->reg0_host);
    const int fw = (p.frame_bits + 31) / 32;
    const size_t smem = sizeof(float2) * (size_t)(T4_THREADS / 32) * 32 * T4F_EROW + 2 * sizeof(uint32_t) * (size_t)p.frames * (fw + 1);
    if (smem > 110 * 1024) return OFDM_OK;            // two CTAs per SM; longer streams take the generic kernel
    p.slot = (const int32_t*)ctx_blob(ctx, slot.data(), sizeof(int32_t) * slot.size());
    p.pilots = (const float2*)ofdm_upload_pilots(ctx, lp->pilot_vals_host, (size_t)lp->Np * lp->S);
    p.tw_t = (const float2*)t4_twiddle_blob(ctx);
    REQUIRE(ctx, p.slot && p.pilots && p.tw_t, "device upload failed");
    CUDA_TRY(ctx, cudaFuncSetAttribute(tx1024_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
    double* part = nullptr;
    if (power) CUDA_TRY(ctx, cudaMallocAsync((void**)&part, sizeof(double) * (size_t)B * p.S, ctx->stream));
    tx1024_kernel<<<(unsigned)B, T4_THREADS, smem, ctx->stream>>>(p, make_devconst<float>(lp->constellation), bits, B * stream_bits, (float2*)time, part);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    int rc = e == cudaSuccess ? OFDM_OK : ctx_fail(ctx, OFDM_ERR_CUDA, "tx1024_kernel launch failed: %s", cudaGetErrorString(e));
    if (rc == OFDM_OK && power) rc = ofdm_power_finish(ctx, part, B, p.S, power);
    if (part) cudaFreeAsync(part, ctx->stream);
    *handled = rc == OFDM_OK;
    return rc;
}

extern "C" int ofdm_cp_autocorr(ofdm_ctx* ctx, const void* rx, int64_t B, int64_t L, int W, int Nfft, void* autocorr, int32_t* tg_pos, double* freq_off,
                                int32_t* fail);

// T4Params of a link with its device tables (0-based carriers, pilots in FP32 and double, twiddles) and the spline plan of
// interp1 over the carriers (no edge extension).  Error messages name the entry point fn.
static int t4_setup(ofdm_ctx* ctx, const char* fn, const ofdm_link_params* lp, int bps, int time_desync, int freq_desync, int mp_desync, T4Params& p,
                    const InterpPlan*& pl) {
    p.Nfft = lp->Nfft; p.logN = ilog2(lp->Nfft); p.Tg = lp->Tg; p.Nc = lp->N_carrier; p.S = lp->S; p.SpF = lp->SpF; p.Nd = lp->Nd; p.Np = lp->Np;
    p.bps = bps; p.scramble = lp->scramble; p.frame_bits = lp->SpF * lp->Nd * bps; p.frames = lp->S / lp->SpF;
    p.time_desync = time_desync != 0; p.freq_desync = freq_desync != 0; p.mp_desync = mp_desync != 0;
    p.prev0 = ofdm_reg_to_prev(lp->reg0_host);
    std::vector<int32_t> d0(lp->Nd), p0(lp->Np);
    for (int i = 0; i < lp->Nd; ++i) {
        if (lp->data_carriers_host[i] < 1 || lp->data_carriers_host[i] > lp->Nfft) return ctx_fail(ctx, OFDM_ERR_INVALID, "%s: data carrier out of range", fn);
        d0[i] = lp->data_carriers_host[i] - 1;
    }
    for (int i = 0; i < lp->Np; ++i) {
        if (lp->pilot_carriers_host[i] < 1 || lp->pilot_carriers_host[i] > lp->N_carrier) return ctx_fail(ctx, OFDM_ERR_INVALID, "%s: pilot carrier out of range", fn);
        if (i > 0 && lp->pilot_carriers_host[i] <= lp->pilot_carriers_host[i - 1]) return ctx_fail(ctx, OFDM_ERR_INVALID, "%s: pilot carriers must increase", fn);
        p0[i] = lp->pilot_carriers_host[i] - 1;
    }
    p.data0 = (const int32_t*)ctx_blob(ctx, d0.data(), sizeof(int32_t) * d0.size());
    p.pil0 = (const int32_t*)ctx_blob(ctx, p0.data(), sizeof(int32_t) * p0.size());
    p.pilots = (const float2*)ofdm_upload_pilots(ctx, lp->pilot_vals_host, (size_t)lp->Np * lp->S);
    p.pilots_d = (const double2*)ctx_blob(ctx, lp->pilot_vals_host, sizeof(double) * 2 * (size_t)lp->Np * lp->S);
    p.tw = (const float2*)ctx_twiddles(ctx, lp->Nfft);
    std::vector<int32_t> q(lp->N_carrier);
    for (int i = 0; i < lp->N_carrier; ++i) q[i] = i + 1;
    pl = ctx_plan(ctx, lp->pilot_carriers_host, lp->Np, 0, q.data(), lp->N_carrier, OFDM_INTERP_SPLINE);
    if (!(p.data0 && p.pil0 && p.pilots && p.pilots_d && p.tw && pl)) return ctx_fail(ctx, OFDM_ERR_INVALID, "%s: device upload failed", fn);
    return OFDM_OK;
}

static const size_t T4_TILES = sizeof(float2) * (T4_THREADS / 32) * 32 * T4F_EROW;   // one 32 x 33 transpose tile per warp
static const int64_t T4_SPLIT_CHUNK = 16384;                   // streams per pass of the split chain: 2.6 GB of kept bins at the Task-4 shape

// dynamic shared memory of t4_post_kernel: region A (angles | rotations | decisions / raw words), then Yp, G, yk, dk
static size_t t4_post_smem(const T4Params& p, const InterpPlan* pl) {
    return (std::max(std::max(sizeof(float) * (size_t)p.S * p.Np, 16 * (size_t)p.Np), std::max(8 * (size_t)T4_THREADS, (size_t)p.S * p.Nd)) + 15) / 16 * 16 +
           sizeof(float2) * ((size_t)p.S * p.Np + p.Nc + 2 * (size_t)pl->n_knots) + 32;
}

typedef void (*t4_post_t)(T4Params, T4FastExtra, PlanDev<float>, DevConst<float>, int64_t, const float2*, const float2*, const uint32_t*, int64_t,
                          uint32_t*, unsigned long long*, double*, double*, float2*, float, T4Stats);

// The split Task-4 chain (Nfft = 1024): t4_ifo_kernel -> t4_sym_kernel -> post, each kernel at its own occupancy, in passes
// of at most T4_SPLIT_CHUNK streams (the caller makes sure an unaligned batch fits one pass).  tg / fo are the detector's
// estimates, ifo is written when the chain corrects the frequency.  post gets the BER outputs (each may be NULL) or, for a
// STATS instantiation, st with its per-stream pointers at stream 0.
static int t4_split_run(ofdm_ctx* ctx, const ofdm_link_params* lp, const T4Params& p, const T4FastExtra& fx, const InterpPlan* pl, t4_post_t post,
                        const void* rx, int64_t B, int64_t L, const int32_t* tg, const double* fo, int32_t* ifo, const uint32_t* tx_bits,
                        uint32_t* out_bits, int64_t* counts, double* tau, double* phase, float2* H, float near_eps, const T4Stats* st) {
    const int64_t CH = std::min<int64_t>(B, T4_SPLIT_CHUNK);
    const int groups = (p.S + T4_THREADS / 32 - 1) / (T4_THREADS / 32);
    const size_t sym_smem = T4_TILES + sizeof(float2) * 1024, post_smem = t4_post_smem(p, pl);
    auto symk = p.Nc <= 416 ? t4_sym_kernel<13> : t4_sym_kernel<32>;
    CUDA_TRY(ctx, cudaFuncSetAttribute(t4_ifo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T4_TILES));
    CUDA_TRY(ctx, cudaFuncSetAttribute(symk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sym_smem));
    CUDA_TRY(ctx, cudaFuncSetAttribute(post, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)post_smem));
    float2* bins = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync((void**)&bins, sizeof(float2) * (size_t)CH * p.S * ((size_t)p.Nd + p.Np), ctx->stream));
    float2* Yd_all = bins;
    float2* Yp_all = bins + (size_t)CH * p.S * p.Nd;
    const int64_t stream_bits = (int64_t)p.frame_bits * p.frames, words = stream_bits / 32;
    int rc = OFDM_OK;
    // (Running the post kernel of one chunk on a side stream under the symbol kernel of the next was tried: the symbol
    // kernel's two CTAs hold every register of an SM, nothing co-resides, and the smaller chunks only add tails.)
    for (int64_t c0 = 0; c0 < B && rc == OFDM_OK; c0 += CH) {
        const int64_t nb = std::min(CH, B - c0);
        const float2* rxc = (const float2*)rx + c0 * L;
        if (p.freq_desync) {
            t4_ifo_kernel<<<(unsigned)cdiv64(nb, T4_THREADS / 32), T4_THREADS, T4_TILES, ctx->stream>>>(fx, rxc, nb, L, p.Tg, p.time_desync, tg + c0, fo + c0, ifo + c0);
            ctx->launches++;
        }
        symk<<<(unsigned)(nb * groups), T4_THREADS, sym_smem, ctx->stream>>>(p, fx, rxc, nb, L, groups, tg + c0, fo + c0, ifo + c0, Yd_all, Yp_all);
        T4Stats s{};
        if (st) {
            s = *st;
            s.rec += c0; s.tg += c0; s.fo += c0; s.ifo += c0; s.nsto += c0; s.cfo += c0;
            if (s.fail) s.fail += c0;
        }
        post<<<(unsigned)nb, T4_THREADS, post_smem, ctx->stream>>>(p, fx, plan_dev<float>(pl), make_devconst<float>(lp->constellation), nb, Yd_all, Yp_all,
                                                                   tx_bits ? tx_bits + c0 * words : nullptr, nb * stream_bits,
                                                                   out_bits ? out_bits + c0 * words : nullptr, (unsigned long long*)counts,
                                                                   tau ? tau + c0 : nullptr, phase ? phase + c0 : nullptr, H ? H + c0 * p.Nc : nullptr, near_eps, s);
        ctx->launches += 2;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "%s launch failed: %s", st ? "statistics chain" : "split Task-4 chain", cudaGetErrorString(e));
    }
    cudaFreeAsync(bins, ctx->stream);
    return rc;
}

extern "C" int ofdm_rx_chain_t4(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx, int64_t B, int time_desync, int freq_desync, int mp_desync,
                                const uint32_t* tx_bits, uint32_t* out_bits, int64_t* counts, int32_t* tg_dev, double* fo_dev, int32_t* ifo_dev,
                                double* tau_dev, double* phase_dev, void* H_dev, double near_eps) {
    return ofdm_rx_chain_t4_ex(ctx, lp, rx, B, time_desync, freq_desync, mp_desync, tx_bits, out_bits, counts, tg_dev, fo_dev, ifo_dev, tau_dev, phase_dev,
                               H_dev, near_eps, nullptr);
}

extern "C" int ofdm_rx_chain_t4_ex(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx, int64_t B, int time_desync, int freq_desync, int mp_desync,
                                   const uint32_t* tx_bits, uint32_t* out_bits, int64_t* counts, int32_t* tg_dev, double* fo_dev, int32_t* ifo_dev,
                                   double* tau_dev, double* phase_dev, void* H_dev, double near_eps, int32_t* fail_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, lp && rx && B >= 0, "bad argument");
    REQUIRE(ctx, ctx->precision == OFDM_PREC_F32, "the fused Task-4 chain is FP32 only (compose the per-function calls in FP64 mode)");
    REQUIRE(ctx, is_pow2(lp->Nfft) && lp->Nfft >= 256 && lp->Nfft <= 2048, "fused Task-4 chain supports Nfft = 256..2048");
    REQUIRE(ctx, lp->S > 0 && lp->SpF > 0 && lp->S % lp->SpF == 0 && lp->Np >= 2 && lp->Nd >= 1 && lp->N_carrier >= 2 && lp->N_carrier <= lp->Nfft, "bad link parameters");
    if (B == 0) return OFDM_OK;
    ConstTable ct = host_constellation(lp->constellation);
    REQUIRE(ctx, ct.bps > 0, "unknown constellation");
    const int64_t L = (int64_t)lp->S * (lp->Nfft + lp->Tg);
    T4Params p;
    const InterpPlan* pl = nullptr;
    int rc = t4_setup(ctx, __func__, lp, ct.bps, time_desync, freq_desync, mp_desync, p, pl);
    if (rc) return rc;
    const int grid = (int)std::min<int64_t>(B, (int64_t)ctx->sm_count * 2);
    // scratch: [estimates: tg int32 | fo double] + per-CTA parking area
    const size_t park = sizeof(float2) * (size_t)grid * lp->S * lp->N_carrier;
    const size_t est = (sizeof(double) + sizeof(int32_t) * 2) * (size_t)B + 64;
    unsigned char* scr = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync((void**)&scr, park + est, ctx->stream));
    double* fo_s = (double*)(scr + park);
    int32_t* tg_s = (int32_t*)(fo_s + B);
    if (!fo_dev) fo_dev = fo_s;
    if (!tg_dev) tg_dev = tg_s;
    if (time_desync || freq_desync) rc = ofdm_cp_autocorr(ctx, rx, B, L, lp->Tg, lp->Nfft, nullptr, tg_dev, fo_dev, fail_dev);
    if (rc == OFDM_OK) {
        const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
        if (out_bits && (stream_bits % 32 != 0 || p.frame_bits % 32 != 0)) {
            cudaError_t e = cudaMemsetAsync(out_bits, 0, sizeof(uint32_t) * OFDM_BIT_WORDS(B * stream_bits), ctx->stream);
            if (e != cudaSuccess) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "memset failed: %s", cudaGetErrorString(e));
        }
        const int fw = (p.frame_bits + 31) / 32;
        size_t smem = sizeof(float2) * (2 * (size_t)p.Nfft + (size_t)p.S * p.Np + p.S + p.Nc + 2 * (size_t)pl->n_knots) + sizeof(double) * (size_t)p.S * p.Np + sizeof(uint32_t) * fw + (size_t)p.SpF * p.Nd + 32;
        // fast path: Nfft = 1024, warp-per-symbol register FFT (rx_t4_fast_kernel)
        bool fast_done = false;
        if (rc == OFDM_OK && p.Nfft == 1024 && !getenv("OFDM_B200_NO_FAST")) {
            const size_t taus = sizeof(double) * (size_t)p.S * p.Np;
            const size_t fsmem = (std::max(T4_TILES, taus) + 15) / 16 * 16 + sizeof(float2) * (1024 + (size_t)p.S * p.Np + p.S + p.Nc + 2 * (size_t)pl->n_knots) + 32;
            if (fsmem <= 111 * 1024 && (size_t)p.S * p.Nd <= std::max(T4_TILES, taus)) {
                T4FastExtra fx;
                fx.tw_t = (const float2*)t4_twiddle_blob(ctx);
                fx.two_a = 2.f * (float)ct.re[12];
                const bool q16 = lp->constellation == OFDM_16QAM, near = near_eps > 0.0, small = p.Nc <= 416;
                typedef void (*kern_t)(T4Params, T4FastExtra, PlanDev<float>, DevConst<float>, const float2*, int64_t, int64_t, const int32_t*, const double*, float2*,
                                       const uint32_t*, int64_t, uint32_t*, unsigned long long*, int32_t*, double*, double*, float2*, float);
                kern_t kern = small ? (q16 ? (near ? rx_t4_fast_kernel<13, true, true> : rx_t4_fast_kernel<13, true, false>)
                                           : (near ? rx_t4_fast_kernel<13, false, true> : rx_t4_fast_kernel<13, false, false>))
                                    : (q16 ? (near ? rx_t4_fast_kernel<32, true, true> : rx_t4_fast_kernel<32, true, false>)
                                           : (near ? rx_t4_fast_kernel<32, false, true> : rx_t4_fast_kernel<32, false, false>));
                // large batches: the same arithmetic as three kernels, each at its own occupancy (t4_split_run)
                const bool aligned = stream_bits % 32 == 0;
                if (fx.tw_t && B >= 512 && (aligned || B <= T4_SPLIT_CHUNK) && t4_post_smem(p, pl) <= 100 * 1024 && p.Np <= T4_THREADS && p.Nd <= p.S * p.Np &&
                    !getenv("OFDM_B200_T4_FUSED")) {
                    int32_t* ifo_ptr = ifo_dev ? ifo_dev : tg_s + B;      // the scratch holds two int32 per stream
                    if (!freq_desync && ifo_dev) cudaMemsetAsync(ifo_dev, 0, sizeof(int32_t) * B, ctx->stream);
                    t4_post_t post = q16 ? (near ? t4_post_kernel<true, true, false> : t4_post_kernel<true, false, false>)
                                         : (near ? t4_post_kernel<false, true, false> : t4_post_kernel<false, false, false>);
                    rc = t4_split_run(ctx, lp, p, fx, pl, post, rx, B, L, tg_dev, fo_dev, ifo_ptr, tx_bits, out_bits, counts, tau_dev, phase_dev, (float2*)H_dev,
                                      (float)near_eps, nullptr);
                    fast_done = true;
                } else if (fx.tw_t) {
                    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem);
                    kern<<<grid, T4_THREADS, fsmem, ctx->stream>>>(p, fx, plan_dev<float>(pl), make_devconst<float>(lp->constellation), (const float2*)rx, B, L, tg_dev, fo_dev,
                                                                   (float2*)scr, tx_bits, B * stream_bits, out_bits, (unsigned long long*)counts, ifo_dev, tau_dev,
                                                                   phase_dev, (float2*)H_dev, (float)near_eps);
                    ctx->launches++;
                    cudaError_t e = cudaGetLastError();
                    if (e != cudaSuccess) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "rx_t4_fast_kernel launch failed: %s", cudaGetErrorString(e));
                    fast_done = true;
                }
            }
        }
        if (rc == OFDM_OK && !fast_done && smem > 200 * 1024) rc = ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "stream shape needs %zu bytes of shared memory", smem);
        if (rc == OFDM_OK && !fast_done) {
            cudaFuncSetAttribute(rx_t4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            rx_t4_kernel<<<grid, T4_THREADS, smem, ctx->stream>>>(p, plan_dev<float>(pl), make_devconst<float>(lp->constellation), (const float2*)rx, B, L, tg_dev, fo_dev,
                                                                   (float2*)scr, tx_bits, B * stream_bits, out_bits, (unsigned long long*)counts, ifo_dev, tau_dev,
                                                                   phase_dev, (float2*)H_dev, (float)near_eps);
            ctx->launches++;
            cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "rx_t4_kernel launch failed: %s", cudaGetErrorString(e));
        }
    }
    cudaFreeAsync(scr, ctx->stream);
    return rc;
}

// Receiver of ofdm_sweep_sync (sweep_sync.cu, not exported): AutoCorrFunction, then the split chain of ofdm_rx_chain_t4_ex
// with t4_post_kernel's STATS instantiation for ANY batch size (ofdm_rx_chain_t4_ex takes it from 512 streams on), so every
// estimate and decision is that of ofdm_rx_chain_t4_ex's split chain on the same streams.  tg / fo / ifo / fail are B-stream
// scratch the call fills; nsto / cfo are the true impairments; Htrue_dev the double N_carrier table; rec the record of the
// first stream (9 fields, stride rec_stride); row the point's counters {errors, bits, detector failures, IFO misses}, +=.
int ofdm_rx_t4_sync_stats(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx, int64_t B, int time_desync, int freq_desync, int mp_desync,
                          const uint32_t* tx_bits, int64_t* row, int32_t* tg, double* fo, int32_t* ifo, int32_t* fail, const int32_t* nsto,
                          const double* cfo, const double* Htrue_dev, double* rec, int64_t rec_stride) {
    REQUIRE(ctx, lp->Nfft == 1024 && ctx->precision == OFDM_PREC_F32, "the statistics chain runs the FP32 Nfft = 1024 kernels");
    REQUIRE(ctx, lp->S > 0 && lp->SpF > 0 && lp->S % lp->SpF == 0 && lp->Np >= 2 && lp->Nd >= 1 && lp->N_carrier >= 2 && lp->N_carrier <= 1024,
            "bad link parameters");
    if (B == 0) return OFDM_OK;
    ConstTable ct = host_constellation(lp->constellation);
    REQUIRE(ctx, ct.bps > 0, "unknown constellation");
    const int64_t L = (int64_t)lp->S * (lp->Nfft + lp->Tg);
    const int64_t stream_bits = (int64_t)lp->S * lp->Nd * ct.bps;
    REQUIRE(ctx, stream_bits % 32 == 0 || B <= T4_SPLIT_CHUNK, "the statistics chain takes at most 16,384 unaligned streams per call");
    T4Params p;
    const InterpPlan* pl = nullptr;
    int rc = t4_setup(ctx, __func__, lp, ct.bps, time_desync, freq_desync, mp_desync, p, pl);
    if (rc) return rc;
    T4FastExtra fx;
    fx.tw_t = (const float2*)t4_twiddle_blob(ctx);
    fx.two_a = 2.f * (float)ct.re[12];
    REQUIRE(ctx, fx.tw_t, "device upload failed");
    // the split-chain conditions of ofdm_rx_chain_t4_ex, each with its own message
    const size_t post_smem = t4_post_smem(p, pl);
    if (post_smem > 100 * 1024) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "stream shape needs %zu bytes of shared memory in the statistics kernel (at most 100 KB)", post_smem);
    if (p.Np > T4_THREADS) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "the statistics chain supports at most %d pilots", T4_THREADS);
    if (p.Nd > p.S * p.Np) return ctx_fail(ctx, OFDM_ERR_UNSUPPORTED, "the statistics chain needs Nd <= S * Np");

    if (time_desync || freq_desync) rc = ofdm_cp_autocorr(ctx, rx, B, L, lp->Tg, 1024, nullptr, tg, fo, fail);
    if (rc) return rc;
    T4Stats st;
    st.Htrue = (const double2*)Htrue_dev; st.rec = rec; st.rec_stride = rec_stride;
    st.tg = tg; st.fo = fo; st.ifo = ifo; st.fail = (time_desync || freq_desync) ? fail : nullptr; st.nsto = nsto; st.cfo = cfo;
    st.a_in = (float)fabs(ct.re[12]); st.a_out = (float)fabs(ct.re[8]);     // 16QAM: re = 1 and 3 (`constellation_func.m`)
    const t4_post_t post = lp->constellation == OFDM_16QAM ? t4_post_kernel<true, false, true> : t4_post_kernel<false, false, true>;
    return t4_split_run(ctx, lp, p, fx, pl, post, rx, B, L, tg, fo, ifo, tx_bits, nullptr, row, nullptr, nullptr, nullptr, 0.f, &st);
}
