// Fast path of the M1 RX chain: Nfft = 4096, N_carrier <= 1024, FP32.
//
// One persistent CTA of 256 threads walks whole streams.  Per OFDM symbol:
//   global -> shared by one 32 KB bulk copy per symbol (TMA engine, CP skipped, two symbols in flight)
//   -> radix-16 pass A in registers -> shared exchange -> pass B -> shared exchange
//   -> pass C pruned to the 1,024 consumed bins (k3 < 4)   [OFDM_demodulator.m:5-8]
//   -> symbol 0 only: pilot LS + edge extension + banded spline operator   [LS_CE.m:27-31]
//   -> one-tap equalise, hard decision, frame-level DeScrambler + BER popcount
//      [equalize_signal.m:6, get_payload.m:3, demapping.m:9-15, DeScrambler.m:8-13, BER_func.m:3]
// Index algebra: n = 256 n1 + 16 n2 + n3, k = k1 + 16 k2 + 256 k3;
//   W4096^{nk} = W16^{n1k1} * W4096^{(16n2+n3)k1} * W16^{n2k2} * W256^{n3k2} * W16^{n3k3}.
// Only outputs k < 1024 are needed, so pass C evaluates 4 of its 16 outputs.
#include "interp.cuh"
#include "fft_reg.cuh"

#define FX_THREADS 256
#define XROW 288          // pass-B output row stride (k1): 16 groups (k2) of 16 samples at stride 18
#define XGRP 18           // ... the two-sample pad per group makes pass C's 128-bit reads conflict free for eight consecutive k2
#define XBUF 4608         // samples per symbol buffer: 16 rows of 288
#define SLOT_ZERO (-2147483647 - 1)

const void* ofdm_upload_pilots(ofdm_ctx* ctx, const double* pv, size_t n_complex);
uint32_t ofdm_reg_to_prev(const uint8_t* reg);


// Cache policy: the symbol stream goes through the copy engine and never touches L1, so what is left of L1 beside
// 2 x 89 KB of shared memory (~55 KB) can hold the channel-estimate tables that every stream re-reads -- provided
// the one-shot traffic (reference bits in, decided bits and H out) does not allocate there.
__device__ __forceinline__ uint32_t ldg_once(const uint32_t* p) {
    uint32_t r;
    asm("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_once(uint32_t* p, uint32_t v) { asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ void stg_once(float2* p, float2 v) { asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory"); }

struct Fast4096Params {
    int Tg, S, SpF, Nc, Nd, Np, frame_words, frames, scramble, con_id;   // frame_words = ceil(frame_bits / 32)
    int txpf;                  // SLIM: prefetch the frame's reference words into L2 (off: OFDM_B200_NO_TXPF)
    int frame_bits, aligned;   // aligned: frame_bits % 32 == 0 (every frame and stream starts on a word of the packed bit arrays)
    uint32_t prev0;
    const int32_t* slot;       // 1024 entries for carriers 0..1023 (data rank / -1-pilot / SLOT_ZERO)
    const float2* pilots;      // Np (first symbol column)
    const float2* tw4096;      // W4096^k
    float inv_sqrt10, two_a;   // 16QAM level unit a = 1/sqrt(10) and the inner decision boundary 2a
};

// ---- mbarrier / bulk-copy (TMA) helpers --------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk async copy global -> shared (TMA engine, SASS UBLKCP), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// L2 prefetch of a block that a later bulk copy will fetch (no shared memory, no completion to wait for)
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Work item q of this CTA = (stream blockIdx.x + (q / S) * gridDim.x, symbol q % S).  Symbols are
// prefetched two items ahead into a two-buffer ring by one elected thread; all three FFT passes run
// in place in the buffer the symbol landed in:
//   pass A  x[256 n1 + t]            -> same places, index k1 replaces n1          (thread-private)
//   pass B  [256 k1 + 16 n2 + n3]    -> [XROW k1 + XGRP k2 + n3]  (XROW 288, XGRP 18: two pad samples per group of 16)
//   pass C  reads 16 consecutive n3 per (k1,k2) as eight 128-bit loads with immediate offsets: conflict-free
//           because of the pad ((9 k2 + j) mod 8 is a permutation over a quarter warp).
// MASK (16 bits, one per k1 = k mod 16): rows of the pass-A output whose carriers {k1 + 16 j} hold no data carrier
// (pilots or unused only).  The channel is estimated from symbol 0 alone (`LS_CE.m:27-28`), so on symbols 1..S-1
// those rows are dead: pass A neither finishes nor stores them and the pass-B warps that own them idle (a comb-4
// layout has MASK 0x1111: a quarter of passes A/B and of their shared-memory traffic).  Symbol 0 runs in full.
__host__ __device__ constexpr int mask_popc(int m) { int n = 0; for (int i = 0; i < 16; ++i) n += (m >> i) & 1; return n; }
// j-th row of the pass-B order: the pruned rows first (so they fill whole warps), then the others, each ascending
__host__ __device__ constexpr int mask_perm(int m, int j) {
    int n = 0;
    for (int i = 0; i < 16; ++i) if ((m >> i) & 1) { if (n == j) return i; ++n; }
    for (int i = 0; i < 16; ++i) if (!((m >> i) & 1)) { if (n == j) return i; ++n; }
    return 0;
}
// SLIM: three CTAs per SM instead of two.  One symbol buffer per CTA (the next symbol is fetched as soon as pass C has read
// the current one, and lands during pass C's arithmetic, the decisions and whatever the two co-resident CTAs are doing) and
// two-level twiddles: W^{t k1} = W^{t (k1 & 3)} * W^{4 t (k1 >> 2)} from six resident values per pass instead of fifteen,
// at the price of nine extra complex multiplications per pass -- 80 registers and 61 KB of shared memory per CTA.
template <bool QAM16, bool NEAR, int MASK, bool SLIM>
__global__ void __launch_bounds__(FX_THREADS, SLIM ? 3 : 2) rx4096_kernel(Fast4096Params p, PlanDev<float> plan, DevConst<float> con, const float2* __restrict__ rx,
                                                               int64_t B, const uint32_t* __restrict__ txbits, uint32_t* __restrict__ outbits,
                                                               float2* __restrict__ Hout, unsigned long long* __restrict__ counts,
                                                               int32_t* __restrict__ err_stream, float near_eps, unsigned long long* __restrict__ next_stream) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bars[2];
    float2* xb0 = (float2*)smem_raw;            // two 4096-sample symbol buffers (ring)
    float2* Hinv = xb0 + (SLIM ? 1 : 2) * XBUF; // 1024
    float2* yk = Hinv + 1024;                   // n_knots
    float2* dk = yk + plan.n_knots;             // n_knots
    int32_t* slot_s = (int32_t*)(dk + plan.n_knots);   // 1024
    float2* pinv = (float2*)(slot_s + 1024);            // Np reciprocals of the first-symbol pilots
    uint8_t* symidx = (uint8_t*)(pinv + p.Np);          // SpF*Nd decisions of the current frame (8-byte aligned)
    const int tid = threadIdx.x;
    const int bps = con.bps;
    for (int i = tid; i < 1024; i += FX_THREADS) slot_s[i] = p.slot[i];
    if (tid < 8) symidx[p.SpF * p.Nd + tid] = 0;          // padding read by the last (partial) word of an unaligned frame
    for (int i = tid; i < p.Np; i += FX_THREADS) { float2 x = p.pilots[i]; float dd = x.x * x.x + x.y * x.y; pinv[i] = make_float2(x.x / dd, -x.y / dd); }

    // per-thread twiddles, resident for the whole kernel.  SLIM keeps W^{t c}, W^{4 t d} (c, d = 1..3) per pass and multiplies
    // twice; the full table is one value per output.
    constexpr int NTW = SLIM ? 4 : 16;
    float2 ta[NTW], tb[NTW];                      // SLIM: [c] = W^{t c}
    float2 ta4[SLIM ? 4 : 1], tb4[SLIM ? 4 : 1];  // SLIM: [d] = W^{4 t d}
#pragma unroll
    for (int k1 = 0; k1 < NTW; ++k1) ta[k1] = p.tw4096[(tid * k1) & 4095];             // W4096^{t*k1}, t = 16 n2 + n3
    {
        const int n3 = tid & 15;
#pragma unroll
        for (int k2 = 0; k2 < NTW; ++k2) tb[k2] = p.tw4096[(16 * n3 * k2) & 4095];     // W256^{n3*k2}
        if (SLIM) {
#pragma unroll
            for (int d = 0; d < 4; ++d) { ta4[d] = p.tw4096[(4 * tid * d) & 4095]; tb4[d] = p.tw4096[(64 * n3 * d) & 4095]; }
        }
    }
    // x * (twiddle of output k = c + 4 d)
    auto twa = [&](float2 x, int c, int d) -> float2 {
        if (SLIM) { if (c) x = cmul(x, ta[c]); if (d) x = cmul(x, ta4[d]); return x; }
        return (c + 4 * d) ? cmul(x, ta[SLIM ? 0 : c + 4 * d]) : x;
    };
    auto twb = [&](float2 x, int c, int d) -> float2 {
        if (SLIM) { if (c) x = cmul(x, tb[c]); if (d) x = cmul(x, tb4[d]); return x; }
        return (c + 4 * d) ? cmul(x, tb[SLIM ? 0 : c + 4 * d]) : x;
    };
    const int symlen = 4096 + p.Tg;
    const int64_t stream_words = (int64_t)p.frame_words * p.frames;
    const float two_a = p.two_a;
    const int64_t my_streams = (B - blockIdx.x + gridDim.x - 1) / gridDim.x;
    const int64_t n_items = my_streams * p.S;
    const int64_t stream_stride = (int64_t)p.S * symlen;                 // samples per stream
    const float2* rx0 = rx + (int64_t)blockIdx.x * stream_stride + p.Tg; // first symbol of this CTA's first stream
    // pass-C coordinates of this thread and its carriers kq + 256 c
    const int k1c = (tid >> 6) + 4 * ((tid >> 3) & 3), k2c = ((tid >> 5) & 1) * 8 + (tid & 7);
    const int kq = k1c + 16 * k2c;
    // pass-B row of this thread and whether its warp owns pruned rows only
    const int k1b = mask_perm(MASK, tid >> 4);
    const bool b_idle = 2 * (tid >> 5) + 1 < mask_popc(MASK);
    // per-thread carrier roles (fixed for the whole kernel): data rank or 0xFFFF, two per register
    uint32_t role01, role23;
    bool warp_data, warp_pil;
    {
        uint32_t r[4];
        bool anyd = false, anyp = false;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int sl = p.slot[kq + 256 * c];
            const bool in = kq + 256 * c < p.Nc;
            r[c] = (sl >= 0 && in) ? (uint32_t)sl : 0xFFFFu;
            anyd |= (sl >= 0 && in);
            anyp |= (sl < 0 && sl != SLOT_ZERO);
        }
        role01 = r[0] | (r[1] << 16); role23 = r[2] | (r[3] << 16);
        warp_data = __any_sync(0xffffffffu, anyd);
        warp_pil = __any_sync(0xffffffffu, anyp);
    }
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // prefetch cursor (used by thread 0 only): item q+2 -> (stream offset, symbol)
    const float2* pf_ptr = rx0;
    int pf_s = 0;
    auto pf_advance = [&]() {
        if (++pf_s == p.S) { pf_s = 0; pf_ptr += (int64_t)gridDim.x * stream_stride - (int64_t)(p.S - 1) * symlen; }
        else pf_ptr += symlen;
    };
    if (tid == 0) {
        for (int i = 0; i < (SLIM ? 1 : 2) && i < n_items; ++i) {
            mbar_expect_tx(&bars[i], 32768u);
            bulk_g2s(xb0 + i * XBUF, pf_ptr, 32768u, &bars[i]);
            pf_advance();
        }
    }
    int errs = 0, nears = 0;
    int s = 0, sf = 0, f = 0;
    int sfNd = 0;                                  // sf * Nd: row of the frame's decision buffer this symbol fills
    int64_t b = blockIdx.x;
    uint32_t parity = 0;
    // SLIM with a scheduling counter: a CTA's first stream is blockIdx.x, every further one is claimed from the counter (no
    // tail: the last streams go to whichever CTAs are free).  The claim for the NEXT stream is made on symbol 0 of the current
    // one, so that the copy / L2 prefetch of its first symbols can be issued on time; all threads pick it up at the stream end.
    __shared__ long long s_bnext[2];                   // double-buffered by stream parity: the next claim never overwrites a slot still being read
    int kpar = 0;
    const bool dyn = SLIM && next_stream != nullptr;
    int64_t bn = dyn ? B : b + gridDim.x;              // thread 0's copy of the next stream (B = none)
    for (int64_t q = 0; dyn ? (b < B) : (q < n_items); ++q) {
        const int cur = SLIM ? 0 : (int)(q & 1);
        float2* X = xb0 + cur * XBUF;
        float2 v[16];
        if (dyn && s == 0 && tid == 0) { bn = (int64_t)gridDim.x + (int64_t)atomicAdd(next_stream, 1ull); s_bnext[kpar] = bn; }
        mbar_wait(&bars[cur], parity);
        parity ^= SLIM ? 1u : (uint32_t)cur;       // flips after every buffer has been used once
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) v[n1] = X[256 * n1 + tid];
        // ---- pass A: DFT over n1 (register index n1 = 4a+b), twiddle W4096^{t*k1}, in place
        const bool pruned = MASK != 0 && s != 0;   // CTA-uniform
        if (pruned) {
            fft16_steps12(v);
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (((MASK >> c) & 0x1111) != 0x1111) fft4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
#pragma unroll
            for (int c = 0; c < 4; ++c)
#pragma unroll
                for (int d = 0; d < 4; ++d) {
                    const int k1 = c + 4 * d;
                    if (!((MASK >> k1) & 1)) X[k1 * 256 + tid] = twa(v[4 * c + d], c, d);
                }
        } else {
            fft16(v);
#pragma unroll
            for (int c = 0; c < 4; ++c)
#pragma unroll
                for (int d = 0; d < 4; ++d) {
                    const int k1 = c + 4 * d;
                    X[k1 * 256 + tid] = twa(v[4 * c + d], c, d);
                }
        }
        __syncthreads();
        // ---- pass B: thread (k1 = k1b, n3 = tid&15), DFT over n2, swizzled write-back; a warp whose two rows are
        // pruned only keeps the barriers company
        const bool b_active = !(pruned && b_idle);
        {
            float2* rp = X + k1b * 256 + (tid & 15);
            if (b_active) {
#pragma unroll
                for (int n2 = 0; n2 < 16; ++n2) v[n2] = rp[16 * n2];
            }
            __syncthreads();                       // every read precedes the swizzled writes
            if (b_active) {
                fft16(v);
                float2* wp = X + k1b * XROW + (tid & 15);
#pragma unroll
                for (int c = 0; c < 4; ++c)
#pragma unroll
                    for (int d = 0; d < 4; ++d) {
                        const int k2 = c + 4 * d;
                        wp[XGRP * k2] = twb(v[4 * c + d], c, d);
                    }
            }
        }
        __syncthreads();
        // ---- pass C: thread (k1c, k2c) -- a quarter warp holds eight consecutive k2 of one k1 (conflict-free 128-bit
        // reads), a warp the four k1 of one residue mod 4 -- DFT over n3, only k3 = 0..3
        {
            const float4* rp = reinterpret_cast<const float4*>(X + k1c * XROW + k2c * XGRP);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 w = rp[j];
                v[2 * j] = make_float2(w.x, w.y);
                v[2 * j + 1] = make_float2(w.z, w.w);
            }
        }
        __syncthreads();                           // buffer `cur` is free: refill it with item q+2
        if (tid == 0 && (SLIM ? (s + 1 < p.S || bn < B) : (q + 2 < n_items))) {
            fence_proxy_async();
            mbar_expect_tx(&bars[cur], 32768u);
            if (SLIM) {     // the item after this one: next symbol of the stream, or symbol 0 of this CTA's next stream (no carried cursor)
                const bool wrap = s + 1 == p.S;
                const float2* nxt = rx + (wrap ? bn : b) * stream_stride + (int64_t)(wrap ? 0 : s + 1) * symlen + p.Tg;
                bulk_g2s(X, nxt, 32768u, &bars[cur]);
                // and the one after that into L2: with a single buffer the copy above is on the critical path
                if (s + 2 < p.S) bulk_prefetch_l2(rx + b * stream_stride + (int64_t)(s + 2) * symlen + p.Tg, 32768u);
                else if (bn < B && s + 2 - p.S < p.S) bulk_prefetch_l2(rx + bn * stream_stride + (int64_t)(s + 2 - p.S) * symlen + p.Tg, 32768u);
            } else {
                bulk_g2s(X, pf_ptr, 32768u, &bars[cur]);
                pf_advance();
            }
        }
        // SLIM has no registers to hold the frame's reference words across pass C: pull them into L2 one symbol before the
        // frame ends instead, so the compare at the frame end waits for L2, not for HBM (16-byte granules only)
        if (SLIM && tid == 0 && txbits && p.txpf && sf == (p.SpF > 1 ? p.SpF - 2 : 0))
            bulk_prefetch_l2(txbits + b * stream_words + (int64_t)f * p.frame_words, (uint32_t)p.frame_words * 4u);
        uint32_t txw[4] = {0u, 0u, 0u, 0u};
        if (!SLIM && sf == p.SpF - 1 && txbits && p.aligned) {  // reference words of this frame, consumed ~400 instructions later
            const uint32_t* tp = txbits + b * stream_words + (int64_t)f * p.frame_words + tid;
#pragma unroll
            for (int j = 0; j < 4; ++j) if (tid + FX_THREADS * j < p.frame_words) txw[j] = ldg_once(tp + FX_THREADS * j);
        }
        // A warp whose carriers are all pilots (comb layouts: the k1 = 0 mod comb rows) has nothing to do after the
        // first symbol of a stream: the channel is estimated from symbol 0 only (`LS_CE.m:27-28`).
        if (warp_data || s == 0) {
            fft16_steps12(v);
            float2 Y[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) Y[c] = add2(add2(v[4 * c], v[4 * c + 1]), add2(v[4 * c + 2], v[4 * c + 3]));   // carrier kq + 256*c
            // ---- symbol 0: LS at the pilots, spline to every carrier, keep 1/H
            if (s == 0) {
                if (warp_pil) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const int sl = slot_s[kq + 256 * c];
                        if (sl < 0 && sl != SLOT_ZERO) { const int pi = -1 - sl; yk[plan.ext_lo + pi] = cmul(Y[c], pinv[pi]); }
                    }
                }
                __syncthreads();
                // Hermite stage: thread tid emits carrier q = tid + 256 u; 1/H goes to the slot of the thread that equalises it
                float2* Hrow = Hout ? Hout + b * p.Nc : nullptr;
                plan_apply_fn<float>(plan, yk, dk, [&](int q, float2 h) {
                    if (Hrow) stg_once(Hrow + q, h);
                    const float dd = h.x * h.x + h.y * h.y;
                    const int k1 = q & 15, k2 = (q >> 4) & 15;
                    Hinv[(((k1 & 3) << 6) | ((k2 >> 3) << 5) | ((k1 >> 2) << 3) | (k2 & 7)) + (q & ~255)] = make_float2(h.x / dd, -h.y / dd);
                });
                __syncthreads();
            }
            // ---- equalise + decide (branch-free per carrier; pilots / unused carriers skip the store)
            if (warp_data) {
                uint8_t* sp = symidx + sfNd;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const uint32_t dr = ((c < 2 ? role01 : role23) >> (16 * (c & 1))) & 0xFFFFu;
                    const float2 e = cmul(Y[c], Hinv[tid + 256 * c]);
                    float margin = 1.f;
                    uint32_t nib;
                    if (QAM16) nib = demap16_nib<NEAR>(e.x, e.y, two_a, &margin);
                    else nib = (uint32_t)nearest_idx(con, e.x, e.y, &margin);
                    // predicated byte store (the decision itself is computed for every lane: no divergent region)
                    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0xFFFF;\n\t@p st.shared.u8 [%1], %2;\n\t}" ::"r"(dr), "r"(smem_u32(sp) + dr), "r"(nib) : "memory");
                    if (NEAR && dr != 0xFFFFu && margin < near_eps) ++nears;
                }
            }
        }
        // ---- frame complete: pack, DeScrambler, compare (reference words were prefetched before pass C's tail)
        if (sf == p.SpF - 1 && !p.aligned) {
            // frames that do not end on a word boundary (e.g. comb 7: 24,556 bits): same packing and descrambling per frame word,
            // the last word masked to the frame, reference bits fetched / decided bits OR-ed in at the frame's bit offset of the
            // packed arrays (out_bits is zeroed by the host entry); the decisions buffer carries eight zero bytes of padding
            __syncthreads();
            const int64_t stream_bits = (int64_t)p.frame_bits * p.frames;
            const int64_t fbase = b * stream_bits + (int64_t)f * p.frame_bits;
            auto packed = [&](int w) -> uint32_t {
                if (QAM16) {
                    const uint2 by = *reinterpret_cast<const uint2*>(symidx + 8 * w);
                    uint32_t lo = by.x | (by.x >> 4); lo = (lo & 0xFFu) | ((lo >> 8) & 0xFF00u);
                    uint32_t hi = by.y | (by.y >> 4); hi = (hi & 0xFFu) | ((hi >> 8) & 0xFF00u);
                    return lo | (hi << 16);
                }
                uint32_t word = 0;
                const int b0 = 32 * w, b1 = min(b0 + 32, p.frame_bits);
                for (int j = b0 / bps; j * bps < b1; ++j) {
                    int idx = symidx[j];
                    for (int i = 0; i < bps; ++i) {
                        int pos = j * bps + i;
                        if (pos >= b0 && pos < b1 && ((idx >> (bps - 1 - i)) & 1)) word |= 1u << (pos - b0);
                    }
                }
                return word;
            };
            for (int w = tid; w < p.frame_words; w += FX_THREADS) {
                const uint32_t cw = packed(w);
                uint32_t o = cw;
                if (p.scramble) { const uint32_t prev = w ? packed(w - 1) : p.prev0; o = cw ^ ((cw << 13) | (prev >> 19)) ^ ((cw << 14) | (prev >> 18)); }
                const int n = min(32, p.frame_bits - 32 * w);
                if (n < 32) o &= (1u << n) - 1u;
                if (txbits) errs += __popc(o ^ bits_get32(txbits, fbase + 32 * (int64_t)w, fbase + p.frame_bits));
                if (outbits) bits_put(outbits, fbase + 32 * (int64_t)w, n, o);
            }
            __syncthreads();                       // the decisions buffer is rewritten by the next frame
        } else if (sf == p.SpF - 1) {
            __syncthreads();
            const int64_t wbase = b * stream_words + (int64_t)f * p.frame_words;
            auto packed = [&](int w) -> uint32_t {
                if (QAM16) {
                    const uint2 by = *reinterpret_cast<const uint2*>(symidx + 8 * w);   // 8 ready-made nibbles, one per byte
                    uint32_t lo = by.x | (by.x >> 4); lo = (lo & 0xFFu) | ((lo >> 8) & 0xFF00u);
                    uint32_t hi = by.y | (by.y >> 4); hi = (hi & 0xFFu) | ((hi >> 8) & 0xFF00u);
                    return lo | (hi << 16);
                }
                uint32_t word = 0;
                const int b0 = 32 * w, b1 = b0 + 32;
                for (int j = b0 / bps; j * bps < b1; ++j) {
                    int idx = symidx[j];
                    for (int i = 0; i < bps; ++i) {
                        int pos = j * bps + i;
                        if (pos >= b0 && pos < b1 && ((idx >> (bps - 1 - i)) & 1)) word |= 1u << (pos - b0);
                    }
                }
                return word;
            };
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int w = tid + FX_THREADS * j;
                if (w < p.frame_words) {
                    const uint32_t cw = packed(w);
                    uint32_t o = cw;
                    if (p.scramble) {
                        const uint32_t prev = w ? packed(w - 1) : p.prev0;
                        o = cw ^ ((cw << 13) | (prev >> 19)) ^ ((cw << 14) | (prev >> 18));
                    }
                    if (txbits) errs += __popc(o ^ (SLIM ? ldg_once(txbits + wbase + w) : txw[j]));
                    if (outbits) stg_once(outbits + wbase + w, o);
                }
            }
            for (int w = tid + 4 * FX_THREADS; w < p.frame_words; w += FX_THREADS) {   // frames longer than 32 Kbit
                const uint32_t cw = packed(w);
                uint32_t o = cw;
                if (p.scramble) { const uint32_t prev = packed(w - 1); o = cw ^ ((cw << 13) | (prev >> 19)) ^ ((cw << 14) | (prev >> 18)); }
                if (txbits) errs += __popc(o ^ txbits[wbase + w]);
                if (outbits) outbits[wbase + w] = o;
            }
        }
        sfNd += p.Nd;
        if (++sf == p.SpF) { sf = 0; sfNd = 0; ++f; }
        if (++s == p.S) {   // stream complete: one atomic per warp that saw errors, no block barrier
            const int we = warp_sum(errs);
            if ((tid & 31) == 0 && we) {
                if (counts) atomicAdd(&counts[0], (unsigned long long)we);
                if (err_stream) atomicAdd(&err_stream[b], we);
            }
            if (NEAR) {
                const int wn = warp_sum(nears);
                if ((tid & 31) == 0 && wn && counts) atomicAdd(&counts[2], (unsigned long long)wn);
            }
            if (tid == 0 && counts) atomicAdd(&counts[1], (unsigned long long)((int64_t)p.frame_bits * p.frames));
            errs = 0; nears = 0; s = 0; sf = 0; sfNd = 0; f = 0;
            if (dyn) { b = s_bnext[kpar]; kpar ^= 1; } else { b += gridDim.x; bn = b + gridDim.x; }
        }
    }
}

int ofdm_rx_chain_fast4096(ofdm_ctx* ctx, const ofdm_link_params* lp, const void* rx, int64_t B, const uint32_t* tx_bits, uint32_t* out_bits,
                           void* H, int64_t* counts, int32_t* err_stream, double near_eps, bool* handled) {
    *handled = false;
    if (ctx->precision != OFDM_PREC_F32 || lp->Nfft != 4096 || lp->N_carrier > 1024 || lp->N_carrier < 2) return OFDM_OK;
    ConstTable ct = host_constellation(lp->constellation);
    if (ct.bps == 0 || lp->S <= 0 || lp->SpF <= 0 || lp->S % lp->SpF) return OFDM_OK;
    const int frame_bits = lp->SpF * lp->Nd * ct.bps;
    if (lp->Np < 2 || lp->Nd < 1) return OFDM_OK;
    if (getenv("OFDM_B200_NO_FAST")) return OFDM_OK;
    std::vector<int32_t> slot(1024, SLOT_ZERO);
    for (int i = 0; i < lp->Nd; ++i) { int c = lp->data_carriers_host[i]; if (c < 1 || c > lp->N_carrier) return OFDM_OK; slot[c - 1] = i; }
    for (int i = 0; i < lp->Np; ++i) {
        int c = lp->pilot_carriers_host[i];
        if (c < 1 || c > lp->N_carrier || (i && c <= lp->pilot_carriers_host[i - 1])) return OFDM_OK;
        slot[c - 1] = -1 - i;
    }
    const InterpPlan* pl = ctx_plan(ctx, lp->pilot_carriers_host, lp->Np, lp->N_carrier, nullptr, lp->N_carrier, OFDM_INTERP_SPLINE);
    REQUIRE(ctx, pl != nullptr, "plan construction failed");
    Fast4096Params p;
    p.Tg = lp->Tg; p.S = lp->S; p.SpF = lp->SpF; p.Nc = lp->N_carrier; p.Nd = lp->Nd; p.Np = lp->Np;
    p.frame_words = (frame_bits + 31) / 32; p.frames = lp->S / lp->SpF; p.scramble = lp->scramble; p.con_id = lp->constellation;
    p.frame_bits = frame_bits; p.aligned = frame_bits % 32 == 0;
    p.txpf = p.aligned && (p.frame_words & 3) == 0 && (((uintptr_t)tx_bits) & 15) == 0 && !getenv("OFDM_B200_NO_TXPF");
    p.prev0 = ofdm_reg_to_prev(lp->reg0_host);
    p.slot = (const int32_t*)ctx_blob(ctx, slot.data(), sizeof(int32_t) * 1024);
    p.pilots = (const float2*)ofdm_upload_pilots(ctx, lp->pilot_vals_host, lp->Np);
    p.tw4096 = (const float2*)ctx_twiddles(ctx, 4096);
    p.inv_sqrt10 = (float)ct.re[12];   // +1/sqrt(10) with the table's own normalisation
    p.two_a = 2.f * p.inv_sqrt10;
    REQUIRE(ctx, p.slot && p.pilots && p.tw4096, "device upload failed");
    if (lp->Tg & 1) return OFDM_OK;          // bulk copies need 16-byte aligned symbol starts
    if (((uintptr_t)rx) & 15) return OFDM_OK;
    size_t smem = sizeof(float2) * (2 * XBUF + 1024 + 2 * (size_t)pl->n_knots) + sizeof(int32_t) * 1024 +
                  (size_t)lp->SpF * lp->Nd + 8 + sizeof(float2) * (size_t)lp->Np + 32;
    if (smem > 110 * 1024) return OFDM_OK;   // keep two CTAs per SM; odd shapes take the generic kernel
    const bool q16 = lp->constellation == OFDM_16QAM;
    const bool near = near_eps > 0.0;
    // rows k1 = k mod 16 of the pass-A output that carry no data carrier: dead after symbol 0
    int dead = 0xFFFF;
    for (int k = 0; k < 1024; ++k) if (slot[k] >= 0) dead &= ~(1 << (k & 15));
    if (getenv("OFDM_B200_NO_PRUNE")) dead = 0;
    typedef void (*kern_t)(Fast4096Params, PlanDev<float>, DevConst<float>, const float2*, int64_t, const uint32_t*, uint32_t*, float2*, unsigned long long*,
                           int32_t*, float, unsigned long long*);
    kern_t kern;
    const size_t smem_slim = smem - sizeof(float2) * XBUF;
    const bool slim = getenv("OFDM_B200_NO_SLIM") == nullptr && smem_slim <= 74 * 1024;
    if (q16 && (dead & 0x1111) == 0x1111) {      // comb 4, 4m
        if (slim) kern = near ? rx4096_kernel<true, true, 0x1111, true> : rx4096_kernel<true, false, 0x1111, true>;
        else kern = near ? rx4096_kernel<true, true, 0x1111, false> : rx4096_kernel<true, false, 0x1111, false>;
    } else if (q16 && (dead & 0x0101) == 0x0101) {   // comb 8, 8m
        if (slim) kern = near ? rx4096_kernel<true, true, 0x0101, true> : rx4096_kernel<true, false, 0x0101, true>;
        else kern = near ? rx4096_kernel<true, true, 0x0101, false> : rx4096_kernel<true, false, 0x0101, false>;
    } else if (q16) {                                // any other 16QAM layout: no dead rows
        if (slim) kern = near ? rx4096_kernel<true, true, 0, true> : rx4096_kernel<true, false, 0, true>;
        else kern = near ? rx4096_kernel<true, true, 0, false> : rx4096_kernel<true, false, 0, false>;
    } else kern = near ? rx4096_kernel<false, true, 0, false> : rx4096_kernel<false, false, 0, false>;
    const bool use_slim = slim && q16;
    if (use_slim) smem = smem_slim;
    CUDA_TRY(ctx, func_smem_optin((const void*)kern, (int)smem));
    int grid = (int)std::min<int64_t>(B, (int64_t)ctx->sm_count * (use_slim ? 3 : 2));
    if (err_stream) CUDA_TRY(ctx, cudaMemsetAsync(err_stream, 0, sizeof(int32_t) * B, ctx->stream));
    if (out_bits && !p.aligned) CUDA_TRY(ctx, cudaMemsetAsync(out_bits, 0, sizeof(uint32_t) * OFDM_BIT_WORDS(B * (int64_t)frame_bits * p.frames), ctx->stream));
    DevConst<float> con = make_devconst<float>(lp->constellation);
    PlanDev<float> pd = plan_dev<float>(pl);
    // the three-CTA kernel claims its streams from a counter (per launch: two launches may be in flight on different streams)
    unsigned long long* sched = nullptr;
    if (use_slim && B > grid && !getenv("OFDM_B200_STATIC_STREAMS")) {
        CUDA_TRY(ctx, cudaMallocAsync((void**)&sched, sizeof(unsigned long long), ctx->stream));
        CUDA_TRY(ctx, cudaMemsetAsync(sched, 0, sizeof(unsigned long long), ctx->stream));
    }
    kern<<<grid, FX_THREADS, smem, ctx->stream>>>(p, pd, con, (const float2*)rx, B, tx_bits, out_bits, (float2*)H, (unsigned long long*)counts, err_stream,
                                                  (float)near_eps, sched);
    if (sched) cudaFreeAsync(sched, ctx->stream);
    LAUNCH_CHECK(ctx);
    *handled = true;
    return OFDM_OK;
}
