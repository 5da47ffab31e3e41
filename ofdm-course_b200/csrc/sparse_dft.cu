// OMP_estimate for partial-DFT dictionaries (`Task 5/OMP_estimate.m:2-37` with the sensing matrix of
// `Task 5/Main_model_Task_5.m:182-190` / `Task5_part2.m:181-190`: A(i,l) = exp(-2*pi*1j*p_i*l/Nfft), p_i = pilot bin, 0-based).
//
// Batch-OMP on the structure of that dictionary -- one correlation per frame instead of one per iteration:
//   * alpha0 = A^H y is one inverse FFT of the measurement scattered onto the pilot bins (SURVEY KAT 6);
//   * the Gram matrix of the dictionary is Toeplitz, (A^H A)[l, c] = g[(l - c) mod Nfft] with
//     g[d] = sum_i exp(+2*pi*1j*p_i*d/Nfft): ONE Nfft-long vector replaces the Ldict x Ldict matrix, so the correlation
//     with the residual r = y - A_S x is  A^H r = alpha0 - sum_q x_q g[(l - c_q) mod Nfft]   (|S| terms per column);
//   * the normal equations of the re-fit (`pinv(A_sel)*y`, :9,17) need only g at the pairwise tap distances and
//     alpha0-like right-hand sides; the stopping rule ||r_i - r_{i-1}|| / ||r_{i-1}|| < 1e-2 (:20) follows from the same
//     Gram quantities (all of that in double, g tabulated in double).
// One CTA per frame; alpha0 lives in registers (16 columns per thread), g in shared memory.  Per frame that is one
// 4096-point FFT + 36 x Ldict complex multiply-adds for K = 9, against 9 x Np x Ldict for the explicit correlations.
// The argmax is taken on FP32 values of alpha; frames whose best two |alpha|^2 differ by less than tie_eps (relative) are
// counted per frame in near_ties (their tap ORDER may differ from a float64 evaluation).
#include "pursuit_common.cuh"
#include "fft_reg.cuh"

#define OD_THREADS 256
#define OD_EPT 16            // dictionary columns per thread: Ldict <= 4096
#define OD_NP_S 256          // measurements staged in shared memory up to this many pilots
#define OD_MAXK 16

// g[d] = sum_i exp(+2*pi*1j*p_i*d/N) = sum_i conj(W_N^{(p_i d) mod N}) from the double twiddle table (exact argument reduction)
__global__ void omp_dft_gram_kernel(const int32_t* __restrict__ p0, int Np, int N, const double2* __restrict__ tw_d, double2* __restrict__ g_d,
                                    float2* __restrict__ g_f) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= N) return;
    double sr = 0, si = 0;
    for (int i = 0; i < Np; ++i) { const double2 w = tw_d[(p0[i] * d) & (N - 1)]; sr += w.x; si -= w.y; }
    g_d[d] = make_double2(sr, si);
    g_f[d] = make_float2((float)sr, (float)si);
}

// Is a dense (Np x Ldict, column-major) dictionary the partial-DFT matrix exp(-2*pi*1j*p_i*l/N) for integer p_i?
// Row i: p_i from the phase of column 1, then every entry is compared.  flag[0] is cleared on the first mismatch.
__global__ void omp_dft_probe_kernel(const float2* __restrict__ A, int Np, int Ldict, int N, int32_t* __restrict__ p0, int32_t* __restrict__ flag) {
    const int i = blockIdx.x;
    __shared__ int sp;
    if (threadIdx.x == 0) {
        const float2 a1 = A[(size_t)Np + i];
        const double turns = -atan2((double)a1.y, (double)a1.x) / (2.0 * CUDART_PI);     // p_i / N mod 1
        int p = (int)llrint(turns * N);
        p &= (N - 1);
        sp = p;
        p0[i] = p;
    }
    __syncthreads();
    const int p = sp;
    bool ok = true;
    for (int l = threadIdx.x; l < Ldict; l += blockDim.x) {
        double s, c;
        sincospi(-2.0 * (double)((p * l) & (N - 1)) / (double)N, &s, &c);
        const float2 a = A[(size_t)l * Np + i];
        if (!(fabs((double)a.x - c) < 2e-6 && fabs((double)a.y - s) < 2e-6)) ok = false;
    }
    if (!ok) atomicAnd(flag, 0);
}

// (best, index, runner-up) merge for the fused argmax + near-tie reduction: first maximum wins (MATLAB max)
struct Top2 { float b1; int i1; float b2; };
__device__ __forceinline__ Top2 top2_merge(Top2 a, Top2 b) {
    Top2 r;
    const bool a_wins = a.b1 > b.b1 || (a.b1 == b.b1 && a.i1 < b.i1);
    if (a_wins) { r.b1 = a.b1; r.i1 = a.i1; r.b2 = fmaxf(a.b2, b.b1); }
    else { r.b1 = b.b1; r.i1 = b.i1; r.b2 = fmaxf(b.b2, a.b1); }
    return r;
}

// Unnormalised inverse 4096-point FFT of fa (natural order) for a 256-thread block: three radix-16 Stockham passes with the
// register butterflies of fft_reg.cuh (forward transform of the conjugate, conjugated on the way out).  Pass 3 leaves
// thread t with the outputs l = t + 256 r in out[r] -- exactly the dictionary columns that thread owns -- so the result never
// goes back to shared memory.  Pass-1 stores (stride 16) are XOR-swizzled within groups of 16 to stay bank-conflict free;
// twiddles W^{q t}, q = 4a + b, are formed as W^{b t} W^{4 a t} from six table reads.  fb is scratch.
__device__ __forceinline__ void od_twiddle16(float2* v, const float2* __restrict__ tw, int t) {
    const float2 b1 = __ldg(tw + t), b2 = __ldg(tw + 2 * t), b3 = __ldg(tw + 3 * t);
    const float2 a1 = __ldg(tw + 4 * t), a2 = __ldg(tw + 8 * t), a3 = __ldg(tw + 12 * t);
    const float2 wb[4] = {make_float2(1.f, 0.f), b1, b2, b3}, wa[4] = {make_float2(1.f, 0.f), a1, a2, a3};
#pragma unroll
    for (int q = 1; q < 16; ++q) {
        const int a = q >> 2, b = q & 3;
        const float2 w = a == 0 ? wb[b] : (b == 0 ? wa[a] : cmul(wb[b], wa[a]));
        v[q] = cmul(v[q], w);
    }
}
__device__ __forceinline__ void od_ifft4096(float2* fa, float2* fb, const float2* __restrict__ tw, int tid, float2* out) {
    float2 v[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) { const float2 x = fa[tid + 256 * q]; v[q] = make_float2(x.x, -x.y); }
    fft16(v);                                            // X[r] sits at v[4 (r & 3) + (r >> 2)]
#pragma unroll
    for (int r = 0; r < 16; ++r) fb[16 * tid + (r ^ (tid & 15))] = v[4 * (r & 3) + (r >> 2)];
    __syncthreads();
    {
        const int k = tid & 15, sw = (tid >> 4) & 15;
#pragma unroll
        for (int q = 0; q < 16; ++q) v[q] = fb[(tid + 256 * q) ^ sw];
        od_twiddle16(v, tw, 16 * k);
        fft16(v);
        float2* o = fa + 16 * tid - 15 * k;
#pragma unroll
        for (int r = 0; r < 16; ++r) o[16 * r] = v[4 * (r & 3) + (r >> 2)];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 16; ++q) v[q] = fa[tid + 256 * q];
    od_twiddle16(v, tw, tid);
    fft16(v);
#pragma unroll
    for (int r = 0; r < 16; ++r) { const float2 x = v[4 * (r & 3) + (r >> 2)]; out[r] = make_float2(x.x, -x.y); }
}

// Warp-wide top-2 of unsigned keys: on return every lane holds the largest key, the smallest index that carries it and the
// largest key among all other candidates (each lane contributes its own runner-up k2 as well).
__device__ __forceinline__ void od_top2_redux(unsigned& k1, int& i1, unsigned& k2) {
    const unsigned K1 = __reduce_max_sync(0xffffffffu, k1);
    const int I1 = (int)__reduce_min_sync(0xffffffffu, k1 == K1 ? (unsigned)i1 : 0x7fffffffu);
    const unsigned K2 = __reduce_max_sync(0xffffffffu, (k1 == K1 && i1 == I1) ? k2 : k1);
    k1 = K1; i1 = I1; k2 = K2;
}

// NG = groups of 256 dictionary columns a thread works on (Ldict <= 256 NG).
//
// The re-fit is carried in ORTHOGONALISED form, so that an iteration needs no triangular solve and the correlation is
// updated in place (only the running alpha lives in registers):
//   u_n = a_{c_n} - sum_{j<n} gamma_jn u_j  = sum_{i<=n} T_in a_{c_i}        (Gram-Schmidt on the selected columns)
//   gamma_jn = u_j^H a_{c_n} / ||u_j||^2 = sum_{i<=j} conj(T_ij) G[c_i][c_n] / ||u_j||^2,   G[c_i][c_n] = g[(c_i - c_n) mod N]
//   beta_n = u_n^H y / ||u_n||^2 = sum_{i<=n} conj(T_in) b_i / ||u_n||^2,     b_i = conj(a_{c_i}) . y
//   r_n = r_{n-1} - u_n beta_n   =>   alpha_n[l] = alpha_{n-1}[l] - sum_{i<=n} (beta_n T_in) g[(l - c_i) mod N]
//   ||r_n - r_{n-1}|| = |beta_n| ||u_n||,  ||r_n||^2 = ||r_{n-1}||^2 - |beta_n|^2 ||u_n||^2      (the stopping rule, :20)
//   x = T beta  is exactly pinv(A_sel) * y  (`OMP_estimate.m:9,17`), formed once at the end.
// All of that is O(k) per lane and iteration, in double; the k+1 coefficients beta_n T_in go to the FP32 update.
template <int NG>
__global__ void __launch_bounds__(OD_THREADS, 3) omp_dft_kernel(const float2* __restrict__ Y, int Np, const int32_t* __restrict__ p0, int Ldict, int Nfft,
                                                                int logN, const float2* __restrict__ tw, const double2* __restrict__ tw_d,
                                                                const float2* __restrict__ g_f, const double2* __restrict__ g_d, int K,
                                                                float2* __restrict__ Hout, float2* __restrict__ hout, int32_t* __restrict__ index_out,
                                                                int32_t* __restrict__ iters_out, int32_t* __restrict__ near_out, float tie_eps) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double red[2 * (OD_THREADS / 32)];
    __shared__ Top2 stop2[OD_THREADS / 32];
    __shared__ int sel[OD_MAXK], ucol[OD_MAXK];
    __shared__ double2 Tm[OD_MAXK][OD_MAXK + 1];      // T[i][n], i <= n
    __shared__ double2 bvec[OD_MAXK], beta[OD_MAXK];
    __shared__ double un2[OD_MAXK], iun2[OD_MAXK];    // ||u_j||^2 and its reciprocal
    __shared__ float2 wf[OD_MAXK], xs[OD_MAXK];
    __shared__ int s_stop;
    __shared__ double s_rr;                            // ||r_{n-1}||^2
    // the per-iteration critical path reads only shared memory: measurements, pilot bins and a two-level double twiddle table
    // W^k = W^{64 (k >> 6)} W^{k & 63} (one double product instead of a gather from the 64 KB global table)
    __shared__ float2 y_s[OD_NP_S];
    __shared__ unsigned short p_s[OD_NP_S];
    __shared__ double2 w_hi[64], w_lo[64];
    __shared__ double2 gcol_s[OD_MAXK], gam_s[OD_MAXK];
    float2* fa = (float2*)smem_raw;
    float2* fb = fa + Nfft;
    const int64_t f = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Nmask = Nfft - 1;
    const float2* y = Y + f * Np;

    // ---- alpha0 = A^H y: scatter onto the pilot bins + unnormalised inverse FFT; ||y||^2 in double
    for (int i = tid; i < Nfft; i += OD_THREADS) fa[i] = make_float2(0.f, 0.f);
    __syncthreads();
    double yy = 0;
    const bool staged = Np <= OD_NP_S;
    for (int i = tid; i < Np; i += OD_THREADS) {
        const float2 v = y[i];
        const int pb = p0[i];
        fa[pb] = v; yy += (double)v.x * v.x + (double)v.y * v.y;
        if (staged) { y_s[i] = v; p_s[i] = (unsigned short)pb; }
    }
    if (tid < 64) { w_hi[tid] = tw_d[(tid * (Nfft >> 6)) & Nmask]; w_lo[tid] = tw_d[tid & Nmask]; }     // Nfft >= 1024: k = (Nfft / 64) a + b, b < Nfft / 64 <= 64
    if (tid == 0) s_stop = 0;
    yy = block_sum(yy, red);          // (barriers inside: the scatter is complete)
    if (tid == 0) s_rr = yy;
    __syncthreads();
    float2 c16[NG == 16 ? 16 : 1];
    float2* c = nullptr;
    if (NG == 16 && Nfft == 4096) od_ifft4096(fa, fb, tw, tid, c16);      // result in registers, in this thread's column order
    else c = block_fft<float, true>(fa, fb, Nfft, logN, tw);
    // the running correlation A^H r, real and imaginary parts of two columns (j, j+1) per register pair: the update below is
    // then four packed FFMA2 per two columns with the tap coefficient as the (hoisted) broadcast operand
    float2 ar[NG / 2], ai[NG / 2];
#pragma unroll
    for (int j = 0; j < NG; j += 2) {
        const int l0 = tid + OD_THREADS * j, l1 = l0 + OD_THREADS;
        float2 c0, c1;
        if (NG == 16 && Nfft == 4096) { c0 = c16[NG == 16 ? j : 0]; c1 = c16[NG == 16 ? j + 1 : 0]; }
        else { c0 = c[l0]; c1 = c[l1 < Nfft ? l1 : l0]; }
        if (l0 >= Ldict) c0 = make_float2(0.f, 0.f);
        if (l1 >= Ldict) c1 = make_float2(0.f, 0.f);
        ar[j / 2] = make_float2(c0.x, c1.x); ai[j / 2] = make_float2(c0.y, c1.y);
    }
    __syncthreads();
    // g twice in a row, real and imaginary planes (both FFT buffers are free now): entry (l - c) mod Nfft is read as
    // gR[base + 256 j] with ONE base per selected tap and immediate offsets, no wrap-around arithmetic in the inner loop
    float* gR = (float*)fa;
    float* gI = gR + 2 * Nfft;
    for (int i = tid; i < 2 * Nfft; i += OD_THREADS) { const float2 v = g_f[i & Nmask]; gR[i] = v.x; gI[i] = v.y; }
    __syncthreads();

    int nu = 0, nsel = 0, near_cnt = 0;                  // block-uniform bookkeeping, carried in registers by every thread
    const bool full_dict = Ldict == OD_THREADS * NG;
    const double g0 = g_d[0].x;                          // ||a_l||^2, the same for every column
    for (int it = 0; it < K; ++it) {
        // ---- first maximum of |A^H r|^2 and the runner-up (`OMP_estimate.m:7,14`).  Per thread: a top-2 scan of its columns in
        // floating point (a NaN never wins a '>').  Across lanes and warps: |.|^2 >= 0, so the IEEE bit pattern + 1 is an
        // order-preserving unsigned key (0 = nothing valid) and each level is three warp-wide REDUX instructions -- largest
        // key, smallest index holding it, largest key among the rest -- instead of five shuffle-and-merge rounds.
        Top2 t; t.b1 = -CUDART_INF_F; t.i1 = 0x7fffffff; t.b2 = -CUDART_INF_F;
        if (full_dict) {
#pragma unroll
            for (int j = 0; j < NG; ++j) {
                const float re = (j & 1) ? ar[j / 2].y : ar[j / 2].x, im = (j & 1) ? ai[j / 2].y : ai[j / 2].x;
                const float m = re * re + im * im;
                if (m > t.b1) { t.b2 = t.b1; t.b1 = m; t.i1 = tid + OD_THREADS * j; } else t.b2 = fmaxf(t.b2, m);
            }
        } else {
#pragma unroll
            for (int j = 0; j < NG; ++j) {
                const int l = tid + OD_THREADS * j;
                const float re = (j & 1) ? ar[j / 2].y : ar[j / 2].x, im = (j & 1) ? ai[j / 2].y : ai[j / 2].x;
                const float m = l < Ldict ? re * re + im * im : -CUDART_INF_F;
                if (m > t.b1) { t.b2 = t.b1; t.b1 = m; t.i1 = l; } else t.b2 = fmaxf(t.b2, m);
            }
        }
        unsigned k1 = t.b1 >= 0.f ? __float_as_uint(t.b1) + 1u : 0u, k2 = t.b2 >= 0.f ? __float_as_uint(t.b2) + 1u : 0u;
        int i1 = t.i1;
        od_top2_redux(k1, i1, k2);
        if (lane == 0) { stop2[warp].b1 = __uint_as_float(k1); stop2[warp].i1 = i1; stop2[warp].b2 = __uint_as_float(k2); }   // keys, bit-cast
        __syncthreads();
        // every warp merges the eight warp results itself (same answer): no warp-0 section, no second barrier
        static_assert(OD_THREADS / 32 == 8, "the final merge assumes eight warps");
        k1 = lane < 8 ? __float_as_uint(stop2[lane & 7].b1) : 0u;
        k2 = lane < 8 ? __float_as_uint(stop2[lane & 7].b2) : 0u;
        i1 = lane < 8 ? stop2[lane & 7].i1 : 0x7fffffff;
        od_top2_redux(k1, i1, k2);
        t.b1 = k1 ? __uint_as_float(k1 - 1u) : -CUDART_INF_F; t.b2 = k2 ? __uint_as_float(k2 - 1u) : -CUDART_INF_F; t.i1 = k1 ? i1 : 0x7fffffff;
        const int col = (t.i1 == 0x7fffffff) ? 0 : t.i1;                  // all-NaN correlation: MATLAB's max returns index 1
        if (!(t.b1 - t.b2 > tie_eps * t.b1)) ++near_cnt;
        const int is_new = __ballot_sync(0xffffffffu, lane < nu && ucol[lane] == col) == 0u;
        if (tid == 0) { sel[nsel] = col; if (is_new) ucol[nu] = col; }     // (readers of the new entry are behind the next barrier)
        ++nsel;
        if (!is_new) break;               // a column selected twice leaves the residual unchanged: ||r_i - r_{i-1}|| = 0 < 1e-2 (`:20`), it >= 1 always here
        // G[c_lane][c_n] for the Gram-Schmidt step below: issued now, consumed after the block-wide b_n (hides the global latency)
        double2 gcol = make_double2(0, 0);
        if (warp == 0 && lane < nu) gcol = g_d[(ucol[lane] - col) & Nmask];
        {
            // b_n = conj(a_new) . y in double, block-wide
            double ar_ = 0, ai_ = 0;
            if (staged) {
                const int qs = logN - 6, qm = (1 << qs) - 1;
                for (int i = tid; i < Np; i += OD_THREADS) {
                    const int k = ((int)p_s[i] * col) & Nmask;
                    const double2 w = cmul(w_hi[k >> qs], w_lo[k & qm]);       // A(i, col)
                    const float2 v = y_s[i];
                    ar_ += w.x * v.x + w.y * v.y; ai_ += w.x * v.y - w.y * v.x;  // conj(w) * v
                }
            } else {
                for (int i = tid; i < Np; i += OD_THREADS) {
                    const double2 w = tw_d[(p0[i] * col) & Nmask];
                    const float2 v = y[i];
                    ar_ += w.x * v.x + w.y * v.y; ai_ += w.x * v.y - w.y * v.x;
                }
            }
            ar_ = warp_sum(ar_); ai_ = warp_sum(ai_);
            if (lane == 0) { red[2 * warp] = ar_; red[2 * warp + 1] = ai_; }
            __syncthreads();
        }
        if (warp == 0) {
            const int n = nu;                                              // index of the new column
            double2 bn = make_double2(0, 0);
            for (int w = 0; w < OD_THREADS / 32; ++w) { bn.x += red[2 * w]; bn.y += red[2 * w + 1]; }
            if (lane == 0) bvec[n] = bn;
            // gamma_j (lane j < n) = sum_{i<=j} conj(T_ij) G[c_i][c_n] / ||u_j||^2   (vectors exchanged through shared memory:
            // independent loads instead of a shuffle per term on the serial path)
            if (lane < n) gcol_s[lane] = gcol;
            __syncwarp();
            double2 gam = make_double2(0, 0);
            if (lane < n) for (int i = 0; i <= lane; ++i) gam = gam + cmul(cconj(Tm[i][lane]), gcol_s[i]);
            const double u2 = lane < n ? un2[lane] : 1.0;
            gam = (lane < n && u2 > 0) ? cscale(gam, iun2[lane]) : make_double2(0, 0);       // iun2 = 1 / ||u_j||^2, kept from iteration j
            if (lane < n) gam_s[lane] = gam;
            __syncwarp();
            // T_in (lane i < n) = - sum_{j=i}^{n-1} gamma_j T_ij ; T_nn = 1
            double2 tin = make_double2(0, 0);
            if (lane < n) for (int j = lane; j < n; ++j) tin = tin - cmul(gam_s[j], Tm[lane][j]);
            if (lane == n) tin = make_double2(1, 0);
            if (lane <= n) Tm[lane][n] = tin;
            // ||u_n||^2 = G_nn - sum_j |gamma_j|^2 ||u_j||^2 ;  beta_n = sum_{i<=n} conj(T_in) b_i / ||u_n||^2
            // (the three warp sums are independent: their shuffle chains overlap)
            double nn = lane < n ? (gam.x * gam.x + gam.y * gam.y) * u2 : 0.0;
            double2 part = make_double2(0, 0);
            if (lane < n) part = cmul(cconj(tin), bvec[lane]);
            else if (lane == n) part = bn;
            nn = warp_sum(nn); part.x = warp_sum(part.x); part.y = warp_sum(part.y);
            const double un = fmax(g0 - nn, 0.0);
            const double iun = un > 0 ? 1.0 / un : 0.0;
            const double2 bt = cscale(part, iun);
            if (lane == 0) { un2[n] = un; iun2[n] = iun; beta[n] = bt; }
            if (lane <= n) { const double2 w = cmul(bt, tin); wf[lane] = make_float2((float)w.x, (float)w.y); }
            // stopping rule: ||r_n - r_{n-1}|| / ||r_{n-1}|| < 1e-2 from the second selection on, compared squared
            // (dn < 1e-4 on: no square roots or division on the serial path; on = 0 never stops, as the quotient form)
            if (lane == 0) {
                const double dn = (bt.x * bt.x + bt.y * bt.y) * un, on = s_rr;
                if (it >= 1 && fmax(dn, 0.0) < 1e-4 * fmax(on, 0.0)) s_stop = 1;
                s_rr = on - dn;
            }
        }
        __syncthreads();
        ++nu;                             // the new column is in
        if (s_stop || it == K - 1) break;
        // ---- alpha -= sum_{i<=n} (beta_n T_in) g[(l - c_i) mod N]
        // (four packed FFMA2 per two columns: the tap coefficient is the hoisted broadcast operand)
        for (int q = 0; q < nu; ++q) {
            const float2 x = wf[q];                                                        // a -= g x:  re -= gr xr - gi xi,  im -= gr xi + gi xr
            const float2 nxr = make_float2(-x.x, -x.x), pxi = make_float2(x.y, x.y), nxi = make_float2(-x.y, -x.y);
            const int base = (tid - ucol[q]) & Nmask;
            const float* gr = gR + base;
            const float* gi = gI + base;
#pragma unroll
            for (int j = 0; j < NG; j += 2) {
                const float2 g_r = make_float2(gr[OD_THREADS * j], gr[OD_THREADS * (j + 1)]);
                const float2 g_i = make_float2(gi[OD_THREADS * j], gi[OD_THREADS * (j + 1)]);
                ar[j / 2] = __ffma2_rn(g_r, nxr, ar[j / 2]);
                ar[j / 2] = __ffma2_rn(g_i, pxi, ar[j / 2]);
                ai[j / 2] = __ffma2_rn(g_r, nxi, ai[j / 2]);
                ai[j / 2] = __ffma2_rn(g_i, nxr, ai[j / 2]);
            }
        }
    }
    __syncthreads();
    // ---- gains x = T beta on the unique columns; a repeated last column shares its unknown (pinv's minimum-norm split)
    __shared__ float2 hval[OD_MAXK];
    if (warp == 0) {
        double2 xv = make_double2(0, 0);
        if (lane < nu) for (int n = lane; n < nu; ++n) xv = xv + cmul(Tm[lane][n], beta[n]);
        const int last = sel[nsel - 1];
        const bool dup = nsel > nu;                      // the last selection repeated column `last`
        if (lane < nu) {
            hval[lane] = (dup && ucol[lane] == last) ? make_float2((float)(0.5 * xv.x), (float)(0.5 * xv.y)) : make_float2((float)xv.x, (float)xv.y);
        }
        __syncwarp();
        if (lane == 0) {
            if (index_out) for (int q = 0; q < K; ++q) index_out[f * K + q] = q < nsel ? sel[q] + 1 : 0;
            if (iters_out) iters_out[f] = nsel;
            if (near_out) near_out[f] = near_cnt;
        }
    }
    __syncthreads();
    if (hout) {
        float2* hb = hout + f * (int64_t)Nfft;
        float4* hb4 = reinterpret_cast<float4*>(hb);
        for (int i = tid; i < Nfft / 2; i += OD_THREADS) hb4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        __syncthreads();                                  // the zeros of this block are ordered before its nu taps
        if (tid < nu) hb[ucol[tid]] = hval[tid];
    }
    if (Hout) {
        // H(m) = sum_u h_u W^{c_u m}; with m = 64 a + b the twiddle is W^{64 c a} * W^{c b}: two 64-entry rows per tap
        float2* t_hi = fb;                       // [nu][64]  h_u * W^{64 c a}
        float2* t_lo = fa;                       // [nu][64]  W^{c b}   (g is no longer needed)
        for (int e = tid; e < nu * 64; e += OD_THREADS) {
            const int u = e >> 6, j = e & 63;
            const float2 v = hval[u];
            const float2 w = tw[(64 * j * ucol[u]) & Nmask];
            t_hi[e] = make_float2(v.x * w.x - v.y * w.y, v.x * w.y + v.y * w.x);
            t_lo[e] = tw[(j * ucol[u]) & Nmask];
        }
        __syncthreads();
        // thread tid owns m = tid + 256 j: b = tid & 63 is fixed (one low twiddle per tap), a = (tid >> 6) + 4 j; NG values of j at a time
        const int bq = tid & 63, a0 = tid >> 6;
        for (int j0 = 0; OD_THREADS * j0 < Nfft; j0 += NG) {
            float2 acc[NG];
#pragma unroll
            for (int j = 0; j < NG; ++j) acc[j] = make_float2(0.f, 0.f);
            for (int u = 0; u < nu; ++u) {
                const float2 w = t_lo[64 * u + bq], wr = make_float2(-w.y, w.x);
                const float2* th = t_hi + 64 * u + a0 + (OD_THREADS / 64) * j0;
#pragma unroll
                for (int j = 0; j < NG; ++j) {
                    const float2 x = th[(OD_THREADS / 64) * j];
                    acc[j] = __ffma2_rn(make_float2(x.x, x.x), w, acc[j]);              // x * w, x the broadcast operand
                    acc[j] = __ffma2_rn(make_float2(x.y, x.y), wr, acc[j]);
                }
            }
#pragma unroll
            for (int j = 0; j < NG; ++j) { const int mm = tid + OD_THREADS * (j0 + j); if (mm < Nfft) Hout[f * (int64_t)Nfft + mm] = acc[j]; }
        }
    }
}

// Batch-OMP path.  p0_dev: Np 0-based pilot bins on the device.  Returns OFDM_OK and sets *handled when it ran.
int ofdm_omp_dft(ofdm_ctx* ctx, const void* y, int64_t B, int Np, const int32_t* p0_dev, int Ldict, int Nfft, int K, void* H, void* h, int32_t* index,
                 int32_t* iters, int32_t* near_ties, double tie_eps, bool* handled) {
    *handled = false;
    if (ctx->precision != OFDM_PREC_F32 || K > OD_MAXK || Ldict > OD_THREADS * OD_EPT || Nfft > 4096 || Nfft < 1024) return OFDM_OK;
    if (getenv("OFDM_B200_NO_BATCH_OMP")) return OFDM_OK;
    const float2* tw = (const float2*)ctx_twiddles(ctx, Nfft);
    const double2* tw_d = (const double2*)ctx_twiddles_prec(ctx, Nfft, OFDM_PREC_F64);
    REQUIRE(ctx, tw != nullptr && tw_d != nullptr, "twiddle allocation failed");
    unsigned char* gbuf = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync((void**)&gbuf, (sizeof(double2) + sizeof(float2)) * (size_t)Nfft, ctx->stream));
    double2* g_d = (double2*)gbuf;
    float2* g_f = (float2*)(g_d + Nfft);
    omp_dft_gram_kernel<<<(Nfft + 63) / 64, 64, 0, ctx->stream>>>(p0_dev, Np, Nfft, tw_d, g_d, g_f);
    const size_t smem = sizeof(float2) * 2 * (size_t)Nfft;
    auto kern = Ldict <= 1024 ? omp_dft_kernel<4> : (Ldict <= 2048 ? omp_dft_kernel<8> : omp_dft_kernel<16>);
    func_smem_optin((const void*)kern, (int)smem);
    kern<<<(unsigned)B, OD_THREADS, smem, ctx->stream>>>((const float2*)y, Np, p0_dev, Ldict, Nfft, ilog2(Nfft), tw, tw_d, g_f, g_d, K, (float2*)H, (float2*)h,
                                                         index, iters, near_ties, (float)tie_eps);
    ctx->launches += 2;
    cudaError_t e = cudaGetLastError();
    cudaFreeAsync(gbuf, ctx->stream);
    if (e != cudaSuccess) return ctx_fail(ctx, OFDM_ERR_CUDA, "Batch-OMP launch failed: %s", cudaGetErrorString(e));
    *handled = true;
    return OFDM_OK;
}

// Dense dictionary: probe for the partial-DFT structure (one 4-byte read-back); on success p0_out (device, Np ints,
// stream-ordered allocation the caller frees) holds the pilot bins.
int ofdm_omp_probe_dft(ofdm_ctx* ctx, const void* A, int Np, int Ldict, int Nfft, int32_t** p0_out, bool* is_dft) {
    *is_dft = false;
    *p0_out = nullptr;
    if (ctx->precision != OFDM_PREC_F32 || Ldict < 2) return OFDM_OK;
    int32_t* buf = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync((void**)&buf, sizeof(int32_t) * ((size_t)Np + 1), ctx->stream));
    int32_t flag = 0;
    CUDA_TRY(ctx, cudaMemsetAsync(buf + Np, 0xFF, sizeof(int32_t), ctx->stream));    // all ones: cleared by the first mismatch
    omp_dft_probe_kernel<<<Np, 128, 0, ctx->stream>>>((const float2*)A, Np, Ldict, Nfft, buf, buf + Np);
    ctx->launches++;
    CUDA_TRY(ctx, cudaMemcpyAsync(&flag, buf + Np, sizeof flag, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (flag != 0) { *is_dft = true; *p0_out = buf; }
    else cudaFreeAsync(buf, ctx->stream);
    return OFDM_OK;
}
