// AutoCorrFunction / remove_IFO / fine_sync -- Task-4 synchronisation on B independent streams.
#include "fft.cuh"
#include <type_traits>

// =====================================================================================
// AutoCorrFunction (`Task 5/AutoCorrFunction.m:1-28`)
// Pass 1: per (stream, tile of outputs) the three sliding-window sums come from one block-wide
// prefix scan held in double (no FP32 cancellation), rho(n) and the "> 0.77 and index > W" flag
// are produced; flags go out as one ballot word per 32 positions.
// Pass 2: one warp per stream finds the first run of consecutive flagged indices, requires a
// second run to exist (else the reference's catch branch: TgPosition = 65), and evaluates
// FreqOffset = -angle(rho(TgPosition))/(2*pi) from a directly summed window.
// =====================================================================================
#define AC_THREADS 128
#define AC_G 16            // samples per group / per thread

// Window sums WITHOUT subtraction (so all-zero windows are exactly 0 and give the reference's 0/0 = NaN, and no
// cancellation error is introduced): with 16-sample groups, the window [n, n+W) starting at n = 16a + r is
//   suffix_a[r] + G[a+1] + ... + G[ge-1] + prefix_ge[oe-1],   ge = (n+W)>>4, oe = (n+W)&15.
// One thread owns one group: it keeps the suffix sums in registers and leaves the prefix sums in shared memory.
template <typename T, bool ALIGNED>
__global__ void __launch_bounds__(AC_THREADS) autocorr_kernel(const cx<T>* __restrict__ rx, int64_t L, int W, int Nfft, int64_t n_out, int tile,
                                                              cx<T>* __restrict__ ac_out, uint32_t* __restrict__ flags, int64_t flag_words,
                                                              const int32_t* __restrict__ gate) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NE = AC_THREADS * AC_G;                 // samples staged per block
    const int PADN = NE + NE / AC_G;                  // one pad word per group: group stride 17 -> conflict-free
    T* Qre = (T*)smem_raw;
    T* Qim = Qre + PADN;
    T* Qa = Qim + PADN;
    T* Qb = Qa + PADN;
    const int64_t b = blockIdx.x;
    if (gate && gate[b] == 0) return;
    const int64_t n0 = (int64_t)blockIdx.y * tile;
    const cx<T>* r = rx + b * L;
    const int tid = threadIdx.x;
    for (int i = tid; i < NE; i += AC_THREADS) {
        const int64_t n = n0 + i;
        cx<T> x = mk<T>(0, 0), y = mk<T>(0, 0);
        if (n + Nfft < L) { x = r[n]; y = r[n + Nfft]; }
        const int q = i + (i >> 4);
        Qre[q] = x.x * y.x + x.y * y.y;               // x * conj(y)
        Qim[q] = x.y * y.x - x.x * y.y;
        Qa[q] = x.x * x.x + x.y * x.y;
        Qb[q] = y.x * y.x + y.y * y.y;
    }
    __syncthreads();
    // own group: suffix sums to registers, prefix sums back to shared memory
    T s0[AC_G], s1[AC_G], s2[AC_G], s3[AC_G];
    {
        const int q0 = tid * (AC_G + 1);
        T v0[AC_G], v1[AC_G], v2[AC_G], v3[AC_G];
#pragma unroll
        for (int i = 0; i < AC_G; ++i) { v0[i] = Qre[q0 + i]; v1[i] = Qim[q0 + i]; v2[i] = Qa[q0 + i]; v3[i] = Qb[q0 + i]; }
        T a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
        for (int i = AC_G - 1; i >= 0; --i) { a0 += v0[i]; a1 += v1[i]; a2 += v2[i]; a3 += v3[i]; s0[i] = a0; s1[i] = a1; s2[i] = a2; s3[i] = a3; }
        a0 = a1 = a2 = a3 = 0;
#pragma unroll
        for (int i = 0; i < AC_G; ++i) { a0 += v0[i]; a1 += v1[i]; a2 += v2[i]; a3 += v3[i]; Qre[q0 + i] = a0; Qim[q0 + i] = a1; Qa[q0 + i] = a2; Qb[q0 + i] = a3; }
    }
    __syncthreads();
    const int wq = W >> 4, wr = W & 15;
    uint32_t mask16 = 0;
    if (tid * AC_G < tile) {
        // groups a+1 .. a+wq-1 are always fully inside the window; group a+wq is inside when r + wr >= 16
        T m0 = 0, m1 = 0, m2 = 0, m3 = 0;
        for (int j = tid + 1; j < tid + wq; ++j) { const int q = j * (AC_G + 1) + AC_G - 1; m0 += Qre[q]; m1 += Qim[q]; m2 += Qa[q]; m3 += Qb[q]; }
        const int qg = (tid + wq) * (AC_G + 1);
        const T g0 = Qre[qg + AC_G - 1], g1 = Qim[qg + AC_G - 1], g2 = Qa[qg + AC_G - 1], g3 = Qb[qg + AC_G - 1];
        const int64_t nb = n0 + tid * AC_G;
        const bool full = (nb + AC_G <= n_out) && (nb + 1 > (int64_t)W);     // uniform for all but the edge groups
#pragma unroll
        for (int rr = 0; rr < AC_G; ++rr) {
            T nr = s0[rr] + m0, ni = s1[rr] + m1, pa = s2[rr] + m2, pb = s3[rr] + m3;
            if (ALIGNED) {                             // W % 16 == 0: the window ends at offset rr of group a + wq
                if (rr > 0) { nr += Qre[qg + rr - 1]; ni += Qim[qg + rr - 1]; pa += Qa[qg + rr - 1]; pb += Qb[qg + rr - 1]; }
            } else {
                int oe = rr + wr;                      // offset of the window end inside its group
                int qt = qg;
                if (oe >= AC_G) { nr += g0; ni += g1; pa += g2; pb += g3; oe -= AC_G; qt += AC_G + 1; }
                if (oe > 0) { nr += Qre[qt + oe - 1]; ni += Qim[qt + oe - 1]; pa += Qa[qt + oe - 1]; pb += Qb[qt + oe - 1]; }
            }
            const int64_t n = nb + rr;
            // |rho| > 0.77  <=>  |num|^2 > 0.77^2 * pa * pb : no division, and 0 > 0 is false exactly where MATLAB's
            // 0/0 = NaN fails the comparison (`AutoCorrFunction.m:6,10-12`)
            const bool above = (nr * nr + ni * ni) > (T)(0.77 * 0.77) * (pa * pb);
            if (above && (full || (n < n_out && n + 1 > (int64_t)W))) mask16 |= 1u << rr;
            if (ac_out && n < n_out) {
                const T den = sqrt(pa * pb);
                ac_out[b * n_out + n] = mk<T>(nr / den, ni / den);   // 0/0 -> NaN as in MATLAB
            }
        }
    }
    const uint32_t hi = __shfl_down_sync(0xffffffffu, mask16, 1);
    if ((tid & 1) == 0 && tid * AC_G < tile) {
        const int64_t wi = (n0 + tid * AC_G) >> 5;
        if (wi < flag_words) flags[b * flag_words + wi] = mask16 | (hi << 16);
    }
}

// FP32 specialisation of the pass above: one float4 {Re num, Im num, |x|^2, |y|^2} per sample in shared memory
// (group stride 17 entries: 128-bit accesses of a quarter warp land in eight different bank groups), packed
// FADD2 for the two pairs.  Same groups, same order of additions, hence the same bits as the generic kernel.
__device__ __forceinline__ float4 f4add(float4 a, float4 b) {
    const float2 lo = __fadd2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y)), hi = __fadd2_rn(make_float2(a.z, a.w), make_float2(b.z, b.w));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}
template <bool ALIGNED>
__global__ void __launch_bounds__(AC_THREADS) autocorr_f32_kernel(const float2* __restrict__ rx, int64_t L, int W, int Nfft, int64_t n_out, int tile,
                                                                  float2* __restrict__ ac_out, uint32_t* __restrict__ flags, int64_t flag_words,
                                                                  const int32_t* __restrict__ list, const int32_t* __restrict__ n_list) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NE = AC_THREADS * AC_G;                 // samples staged per block
    float4* Q = (float4*)smem_raw;                    // NE + NE/16 entries
    // `list` (second, full-length scan): blockIdx.x is a slot that walks the streams the prefix scan left unresolved -- a
    // handful at most, so the grid is a few hundred slots instead of one CTA per stream and tile
    const int n_it = list ? *n_list : 1;
    for (int it = list ? (int)blockIdx.x : 0; it < n_it; it += list ? (int)gridDim.x : 1) {
    const int64_t b = list ? list[it] : blockIdx.x;
    const int64_t n0 = (int64_t)blockIdx.y * tile;
    const float2* r = rx + b * L;
    const int tid = threadIdx.x;
    // staging: sample n0 + 128 j + tid and its partner one FFT length later, all loads of a thread in flight at once
    {
        float2 x[AC_G], y[AC_G];
        const float2* rp = r + n0 + tid;
        if (n0 + NE + Nfft <= L) {                    // interior tile: no bounds checks
#pragma unroll
            for (int j = 0; j < AC_G; ++j) { x[j] = __ldg(rp + AC_THREADS * j); y[j] = __ldg(rp + AC_THREADS * j + Nfft); }
        } else {
#pragma unroll
            for (int j = 0; j < AC_G; ++j) {
                const bool ok = n0 + tid + AC_THREADS * j + Nfft < L;
                x[j] = ok ? __ldg(rp + AC_THREADS * j) : make_float2(0.f, 0.f);
                y[j] = ok ? __ldg(rp + AC_THREADS * j + Nfft) : make_float2(0.f, 0.f);
            }
        }
#pragma unroll
        for (int j = 0; j < AC_G; ++j) {
            const int i = tid + AC_THREADS * j;
            Q[i + (i >> 4)] = make_float4(x[j].x * y[j].x + x[j].y * y[j].y, x[j].y * y[j].x - x[j].x * y[j].y, x[j].x * x[j].x + x[j].y * x[j].y,
                                          y[j].x * y[j].x + y[j].y * y[j].y);   // x * conj(y), |x|^2, |y|^2
        }
    }
    __syncthreads();
    float4 sfx[AC_G];                                 // suffix sums of the own group
    {
        const int q0 = tid * (AC_G + 1);
        float4 v[AC_G];
#pragma unroll
        for (int i = 0; i < AC_G; ++i) v[i] = Q[q0 + i];
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = AC_G - 1; i >= 0; --i) { a = f4add(a, v[i]); sfx[i] = a; }
        a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < AC_G; ++i) { a = f4add(a, v[i]); Q[q0 + i] = a; }    // prefix sums back to shared memory
    }
    __syncthreads();
    const int wq = W >> 4, wr = W & 15;
    uint32_t mask16 = 0;
    if (tid * AC_G < tile) {
        float4 m = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = tid + 1; j < tid + wq; ++j) m = f4add(m, Q[j * (AC_G + 1) + AC_G - 1]);
        const int qg = (tid + wq) * (AC_G + 1);
        const float4 g = Q[qg + AC_G - 1];
        const int64_t nb = n0 + tid * AC_G;
        const bool full = (nb + AC_G <= n_out) && (nb + 1 > (int64_t)W);
#pragma unroll
        for (int rr = 0; rr < AC_G; ++rr) {
            float4 t = f4add(sfx[rr], m);
            if (ALIGNED) {
                if (rr > 0) t = f4add(t, Q[qg + rr - 1]);
            } else {
                int oe = rr + wr;
                int qt = qg;
                if (oe >= AC_G) { t = f4add(t, g); oe -= AC_G; qt += AC_G + 1; }
                if (oe > 0) t = f4add(t, Q[qt + oe - 1]);
            }
            const bool above = (t.x * t.x + t.y * t.y) > (float)(0.77 * 0.77) * (t.z * t.w);
            if (above) mask16 |= 1u << rr;
            if (ac_out) {
                const int64_t n = nb + rr;
                if (n < n_out) {
                    const float den = sqrtf(t.z * t.w);
                    ac_out[b * n_out + n] = make_float2(t.x / den, t.y / den);   // 0/0 -> NaN as in MATLAB
                }
            }
        }
        if (!full) {                                   // edge groups: drop positions outside (W, n_out]
            uint32_t keep = 0;
#pragma unroll
            for (int rr = 0; rr < AC_G; ++rr) { const int64_t n = nb + rr; if (n < n_out && n + 1 > (int64_t)W) keep |= 1u << rr; }
            mask16 &= keep;
        }
    }
    const uint32_t hi = __shfl_down_sync(0xffffffffu, mask16, 1);
    if ((tid & 1) == 0 && tid * AC_G < tile) {
        const int64_t wi = (n0 + tid * AC_G) >> 5;
        if (wi < flag_words) flags[b * flag_words + wi] = mask16 | (hi << 16);
    }
    if (list) __syncthreads();                        // the staging area is reused by the slot's next stream
    }
}

template <typename T>
__global__ void autocorr_detect_kernel(const cx<T>* __restrict__ rx, int64_t B, int64_t L, int W, int Nfft, int64_t n_out,
                                       const uint32_t* __restrict__ flags, int64_t flag_words, int32_t* __restrict__ tg_pos,
                                       double* __restrict__ freq_off, int32_t* __restrict__ fail, const int32_t* __restrict__ gate,
                                       int32_t* __restrict__ list, int32_t* __restrict__ n_list) {
    const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (b >= B) return;
    if (gate && gate[b] == 0) return;
    const uint32_t* fw = flags + b * flag_words;
    const int BIG = 0x7fffffff;
    // first flagged index
    int f = BIG;
    for (int64_t wi = lane; wi < flag_words; wi += 32) { uint32_t x = fw[wi]; if (x) { f = (int)(wi * 32 + __ffs(x) - 1); break; } }
    f = warp_min(f);
    int e = BIG, g = BIG;
    if (f != BIG) {
        // first un-flagged index after f (positions >= n_out count as un-flagged)
        for (int64_t wi = (f >> 5) + ((lane - ((f >> 5) & 31)) & 31); wi < flag_words; wi += 32) {
            uint32_t x = ~fw[wi];
            if (wi == (f >> 5)) x &= ~((2u << (f & 31)) - 1u);   // only positions > f
            if (x) { e = (int)(wi * 32 + __ffs(x) - 1); break; }
        }
        e = warp_min(e);
        if (e == BIG || e > n_out) e = (int)n_out;
        // any flagged index after e -> a second run exists (`result(2)` is defined)
        for (int64_t wi = (e >> 5) + ((lane - ((e >> 5) & 31)) & 31); wi < flag_words; wi += 32) {
            uint32_t x = fw[wi];
            if (wi == (e >> 5)) x &= ~((1u << (e & 31)) - 1u);   // positions >= e (e itself is clear)
            if (x) { g = (int)(wi * 32 + __ffs(x) - 1); break; }
        }
        g = warp_min(g);
    }
    int tg = 65, failed = 1;
    if (f != BIG && g != BIG) { tg = (f + 1 + e) / 2; failed = 0; }   // floor((first+last)/2), 1-based
    // rho(TgPosition) summed directly in double
    double nr = 0, ni = 0, pa = 0, pb = 0;
    const int64_t n = tg - 1;
    if (n < n_out) {
        const cx<T>* r = rx + b * L;
        for (int k = lane; k < W; k += 32) {
            cx<T> x = r[n + k], y = r[n + k + Nfft];
            double xr = x.x, xi = x.y, yr = y.x, yi = y.y;
            nr += xr * yr + xi * yi; ni += xi * yr - xr * yi; pa += xr * xr + xi * xi; pb += yr * yr + yi * yi;
        }
        nr = warp_sum(nr); ni = warp_sum(ni); pa = warp_sum(pa); pb = warp_sum(pb);
    } else { nr = ni = CUDART_NAN; }
    if (lane == 0) {
        double den = sqrt(pa * pb);
        tg_pos[b] = tg;
        freq_off[b] = -atan2(ni / den, nr / den) / (2.0 * CUDART_PI);
        if (fail) fail[b] = failed;
        if (list && failed) list[atomicAdd(n_list, 1)] = (int32_t)b;      // prefix scan: unresolved streams for the full-length pass
    }
}

extern "C" int ofdm_cp_autocorr(ofdm_ctx* ctx, const void* rx, int64_t B, int64_t L, int W, int Nfft, void* autocorr,
                                int32_t* tg_pos, double* freq_off, int32_t* fail) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, rx && tg_pos && freq_off && B >= 0 && W > 0 && Nfft > 0, "bad argument");
    const int64_t n_out = L - W - Nfft;
    REQUIRE(ctx, n_out >= 65, "stream too short for AutoCorrFunction (needs L-W-Nfft >= 65)");
    REQUIRE(ctx, W <= 1536, "window wider than 1536 samples (the tile of 16*(126 - W/16) outputs per block must stay positive)");
    if (B == 0) return OFDM_OK;
    REQUIRE(ctx, W >= AC_G, "window narrower than 16 samples");
    // outputs per block: every output needs groups a .. a + W/16 + 1 staged; keep the group count even (32-bit flag words)
    const int tile = AC_G * ((AC_THREADS - (W >> 4) - 2) & ~1);
    // When the AutoCorr vector itself is not wanted, TgPosition is decided by the first run of indices above the threshold
    // and by the mere EXISTENCE of a second run (`AutoCorrFunction.m:15-20`), which normally starts one symbol later.  So the
    // first three symbol lengths are scanned first; a stream whose prefix already holds "first run, gap, flagged index" has
    // exactly the result of the full scan, every other stream (fail flag set) is re-scanned at full length by gated kernels.
    const int64_t n_prefix = cdiv64(3 * (int64_t)(Nfft + W), tile) * tile;
    const bool two_stage = autocorr == nullptr && n_prefix < n_out && !getenv("OFDM_B200_FULL_AUTOCORR");
    const int64_t flag_words = (n_out + 31) / 32;
    uint32_t* flags = (uint32_t*)ctx_scratch(ctx, sizeof(uint32_t) * B * flag_words + sizeof(int32_t) * (2 * B + 1) + 64);
    REQUIRE(ctx, flags != nullptr, "scratch allocation failed");
    int32_t* fail_s = (int32_t*)(flags + B * flag_words);
    int32_t* list = fail_s + B;                           // unresolved streams of the prefix scan, then their count
    int32_t* n_list = list + B;
    if (two_stage && !fail) fail = fail_s;
    if (two_stage) CUDA_TRY(ctx, cudaMemsetAsync(n_list, 0, sizeof(int32_t), ctx->stream));
    for (int stage = two_stage ? 0 : 1; stage < 2; ++stage) {
        const int64_t n_scan = stage == 0 ? n_prefix : n_out;
        const int64_t fw = (n_scan + 31) / 32;
        const int tiles = (int)cdiv64(n_scan, tile);
        const bool second = two_stage && stage == 1;
        const int32_t* gate = second ? fail : nullptr;
        DISPATCH_T(ctx, {
            size_t smem = 4 * sizeof(T) * (size_t)(AC_THREADS * AC_G + AC_THREADS);
            if constexpr (std::is_same<T, float>::value) {
                auto k1 = (W & 15) ? autocorr_f32_kernel<false> : autocorr_f32_kernel<true>;
                const unsigned gx = second ? (unsigned)std::min<int64_t>(B, 256) : (unsigned)B;
                k1<<<dim3(gx, tiles), AC_THREADS, smem, ctx->stream>>>((const float2*)rx, L, W, Nfft, n_scan, tile, (float2*)autocorr, flags, fw,
                                                                        second ? list : nullptr, second ? n_list : nullptr);
            } else {
                auto k1 = (W & 15) ? autocorr_kernel<T, false> : autocorr_kernel<T, true>;
                if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k1, (int)smem));
                k1<<<dim3((unsigned)B, tiles), AC_THREADS, smem, ctx->stream>>>((const cx<T>*)rx, L, W, Nfft, n_scan, tile, (cx<T>*)autocorr, flags, fw, gate);
            }
            ctx->launches++;
            autocorr_detect_kernel<T><<<(unsigned)cdiv64(B * 32, 128), 128, 0, ctx->stream>>>((const cx<T>*)rx, B, L, W, Nfft, n_scan, flags, fw,
                                                                                                tg_pos, freq_off, fail, gate,
                                                                                                (two_stage && stage == 0) ? list : nullptr, n_list);
        });
        LAUNCH_CHECK(ctx);
    }
    return OFDM_OK;
}

// =====================================================================================
// remove_IFO (`Task 5/remove_IFO.m:1-11`): first bin of abs(fft(rx(Nfft+1:2*Nfft))) above 0.77,
// then add_CFO(rx, -IFO, Nfft) with the exact integer phase (IFO*n mod Nfft) from the twiddle table.
// =====================================================================================
template <typename T>
__global__ void ifo_detect_kernel(const cx<T>* __restrict__ rx, int64_t L, int N, int logN, const cx<T>* __restrict__ tw,
                                  int32_t* __restrict__ ifo) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int red[32];
    using C = cx<T>;
    C* a = (C*)smem_raw;
    C* bb = a + N;
    const int64_t b = blockIdx.x;
    const C* src = rx + b * L + N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) a[i] = src[i];
    __syncthreads();
    C* r = block_fft<T, false>(a, bb, N, logN, tw);
    int first = 0x7fffffff;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        double re = r[i].x, im = r[i].y;
        if (sqrt(re * re + im * im) > 0.77) { first = i; break; }   // strided ascending: first hit per thread is its minimum
    }
    first = block_min(first, red);
    if (threadIdx.x == 0) ifo[b] = (first == 0x7fffffff) ? -1 : first;
}
template <typename T>
__global__ void ifo_derotate_kernel(const cx<T>* __restrict__ rx, int64_t B, int64_t L, int N, const cx<T>* __restrict__ tw,
                                    const int32_t* __restrict__ ifo, cx<T>* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * L) return;
    int64_t b = i / L, n = i - b * L;
    int k = ifo[b];
    cx<T> v = rx[i];
    if (k > 0) v = cmul(v, tw[(int)(((int64_t)k * n) & (N - 1))]);   // exp(-2j*pi*IFO*n/Nfft)
    out[i] = v;
}
extern "C" int ofdm_remove_ifo(ofdm_ctx* ctx, const void* rx, int64_t B, int64_t L, int Nfft, void* out, int32_t* ifo) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, rx && out && ifo && B >= 0, "bad argument");
    REQUIRE(ctx, is_pow2(Nfft) && Nfft >= 8 && Nfft <= (ctx->precision == OFDM_PREC_F64 ? 4096 : 8192), "unsupported Nfft");
    REQUIRE(ctx, L >= 2 * (int64_t)Nfft, "stream shorter than 2*Nfft");
    if (B == 0) return OFDM_OK;
    const void* tw = ctx_twiddles(ctx, Nfft);
    REQUIRE(ctx, tw != nullptr, "twiddle allocation failed");
    DISPATCH_T(ctx, {
        size_t smem = 2 * (size_t)Nfft * sizeof(cx<T>);
        auto k1 = ifo_detect_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k1, (int)smem));
        k1<<<(unsigned)B, fft_threads(Nfft), smem, ctx->stream>>>((const cx<T>*)rx, L, Nfft, ilog2(Nfft), (const cx<T>*)tw, ifo);
        ctx->launches++;
        ifo_derotate_kernel<T><<<(unsigned)cdiv64(B * L, 256), 256, 0, ctx->stream>>>((const cx<T>*)rx, B, L, Nfft, (const cx<T>*)tw, ifo, (cx<T>*)out);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}

// =====================================================================================
// fine_sync (`Task 4/fine_sync.m:1-60`).  Estimators run in double on the (T-typed) pilots.
// =====================================================================================
#define FS_THREADS 256
template <typename T>
__global__ void __launch_bounds__(FS_THREADS) fine_sync_est_kernel(const cx<T>* __restrict__ grid, int S, int Nfft, const int32_t* __restrict__ pc0,
                                                                   int Np, const double2* __restrict__ txp /* Np x S col-major */, int time_desync,
                                                                   double* __restrict__ tau_out, double* __restrict__ phase_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* taus = (double*)smem_raw;       // M-1 entries
    __shared__ int cnt[FS_THREADS];
    __shared__ double red[32];
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x;
    const int M = Np * S;
    const cx<T>* g = grid + b * (int64_t)S * Nfft;
    const double deltak = (double)(pc0[1] - pc0[0]);                     // :6
    auto q_at = [&](int i) -> double2 {                                   // tx * conj(rx), column-major flat index
        int s = i / Np, p = i - s * Np;
        double2 rxv = to_d(g[(int64_t)s * Nfft + pc0[p]]);
        return cmulc(txp[i], rxv);
    };
    for (int j = tid; j < M - 1; j += FS_THREADS) {                        // taus(j+1) in MATLAB terms (:25-30)
        double2 q1 = q_at(j + 1), q0 = q_at(j);
        double2 d = cmulc(q1, q0);
        taus[j] = atan2(d.y, d.x) / (2.0 * CUDART_PI * deltak);
    }
    __syncthreads();
    // mask = [false, abs(diffs)<1e-3 & abs(diffs)~=0]; taus_result = taus(mask); mean(taus_result(Np+1:end))
    const int n = M - 1;
    const int CH = (n + FS_THREADS - 1) / FS_THREADS;
    const int lo = min(tid * CH, n), hi = min(lo + CH, n);
    int c = 0;
    for (int j = max(lo, 1); j < hi; ++j) { double d = fabs(taus[j] - taus[j - 1]); c += (d < 1e-3 && d != 0.0); }
    int rank = block_exclusive_scan(c, cnt);            // survivors before this thread's chunk
    double sum = 0; int kept = 0;
    for (int j = max(lo, 1); j < hi; ++j) {
        double d = fabs(taus[j] - taus[j - 1]);
        if (d < 1e-3 && d != 0.0) { if (rank >= Np) { sum += taus[j]; ++kept; } ++rank; }
    }
    sum = block_sum(sum, red);
    double nk = block_sum((double)kept, red);
    const double tau = sum / nk;                                            // empty -> NaN like mean([])
    // common phase after the (optional) timing correction (:47-52)
    double ps = 0; int pn = 0;
    for (int i = tid; i < M; i += FS_THREADS) {
        int s = i / Np, p = i - s * Np;
        double2 rxv = to_d(g[(int64_t)s * Nfft + pc0[p]]);
        if (time_desync) { double sn, cs; sincospi(2.0 * tau * (double)pc0[p], &sn, &cs); rxv = cmul(rxv, make_double2(cs, sn)); }
        double2 qq = cmulc(txp[i], rxv);
        double a = atan2(qq.y, qq.x);
        if (fabs(a) > 1e-3) { ps += a; ++pn; }
    }
    ps = block_sum(ps, red);
    double pk = block_sum((double)pn, red);
    if (tid == 0) { tau_out[b] = tau; phase_out[b] = ps / pk; }
}
template <typename T>
__global__ void fine_sync_apply_kernel(const cx<T>* __restrict__ grid, int64_t B, int S, int Nfft, const double* __restrict__ tau,
                                       const double* __restrict__ phase, int time_desync, int freq_desync, cx<T>* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * S * (int64_t)Nfft) return;
    int n = (int)(i % Nfft);
    int64_t b = i / ((int64_t)S * Nfft);
    double2 v = to_d(grid[i]);
    if (time_desync) { double sn, cs; sincospi(2.0 * tau[b] * (double)n, &sn, &cs); v = cmul(v, make_double2(cs, sn)); }  // nn_exp' = exp(+2j*pi*tau*n)
    if (freq_desync) { double sn, cs; sincos(phase[b], &sn, &cs); v = cmul(v, make_double2(cs, sn)); }
    out[i] = from_d<T>(v);
}

const void* ofdm_upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex);

extern "C" int ofdm_fine_sync(ofdm_ctx* ctx, const void* grid, int64_t B, int S, int Nfft, const int32_t* pc, int Np, const double* pv,
                              int time_desync, int freq_desync, void* out, double* tau_dev, double* phase_dev) {
    if (!ctx) return OFDM_ERR_INVALID;
    REQUIRE(ctx, grid && out && pc && pv && B >= 0 && S > 0 && Np >= 2, "bad argument");
    if (B == 0) return OFDM_OK;
    std::vector<int32_t> p0(Np);
    for (int i = 0; i < Np; ++i) { REQUIRE(ctx, pc[i] >= 1 && pc[i] <= Nfft, "pilot index out of range"); p0[i] = pc[i] - 1; }
    const int32_t* pc0 = (const int32_t*)ctx_blob(ctx, p0.data(), sizeof(int32_t) * Np);
    const double2* txp = (const double2*)ctx_blob(ctx, pv, sizeof(double) * 2 * (size_t)Np * S);
    REQUIRE(ctx, pc0 && txp, "device upload failed");
    double* est = nullptr;
    if (!tau_dev || !phase_dev) {
        est = (double*)ctx_scratch(ctx, sizeof(double) * 2 * B);
        REQUIRE(ctx, est != nullptr, "scratch allocation failed");
        if (!tau_dev) tau_dev = est;
        if (!phase_dev) phase_dev = est + B;
    }
    size_t smem = sizeof(double) * (size_t)(Np * S);
    DISPATCH_T(ctx, {
        auto k1 = fine_sync_est_kernel<T>;
        if (smem > 48 * 1024) CUDA_TRY(ctx, func_smem_optin((const void*)k1, (int)smem));
        k1<<<(unsigned)B, FS_THREADS, smem, ctx->stream>>>((const cx<T>*)grid, S, Nfft, pc0, Np, txp, time_desync, tau_dev, phase_dev);
        ctx->launches++;
        int64_t n = B * S * (int64_t)Nfft;
        fine_sync_apply_kernel<T><<<(unsigned)cdiv64(n, 256), 256, 0, ctx->stream>>>((const cx<T>*)grid, B, S, Nfft, tau_dev, phase_dev, time_desync,
                                                                                       freq_desync, (cx<T>*)out);
    });
    LAUNCH_CHECK(ctx);
    return OFDM_OK;
}
