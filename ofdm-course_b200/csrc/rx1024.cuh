// Per-symbol device code of the Nfft = 1024 receivers shared by the Task-4 chain (chain_rx_t4.cu) and the one-pass Task-3
// receiver of ofdm_sweep_mer (sweep_mer.cu): the symbol window load, the first pass of the warp-per-symbol 1024-point
// transform, and the 16QAM MER term.  One copy, so both receivers compute bit-identical bins and MER sums.
#pragma once
#include "fft_reg.cuh"

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
const void* t4_twiddle_blob(ofdm_ctx* ctx);                 // the tw_t table (chain_rx_t4.cu)

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

// 16QAM point nearest to e, per axis (the separable rule of demap16_nib), accumulated as `MER_func.m:7-25` does.  It is the
// point MER_func's abs() search returns except for exact ties on a decision boundary, where either point is equally near.
__device__ __forceinline__ void t4_mer16(float2 e, float two_a, float a_in, float a_out, double& s1, double& s2) {
    const float ix = copysignf(fabsf(e.x) < two_a ? a_in : a_out, e.x), iy = copysignf(fabsf(e.y) < two_a ? a_in : a_out, e.y);
    const double er = (double)ix - (double)e.x, ei = (double)iy - (double)e.y;
    s1 += (double)ix * ix + (double)iy * iy;
    s2 += er * er + ei * ei;
}
