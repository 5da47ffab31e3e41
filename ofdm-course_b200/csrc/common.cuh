// Shared device/host helpers of libofdm_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/ofdm_b200.h"

// ------------------------------------------------------------------ complex helpers
template <typename T> struct cplx;
template <> struct cplx<float> { using type = float2; };
template <> struct cplx<double> { using type = double2; };
template <typename T> using cx = typename cplx<T>::type;

template <typename T> __host__ __device__ __forceinline__ cx<T> mk(T a, T b) { cx<T> r; r.x = a; r.y = b; return r; }
__host__ __device__ __forceinline__ float2 operator+(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__host__ __device__ __forceinline__ float2 operator-(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__host__ __device__ __forceinline__ double2 operator+(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__host__ __device__ __forceinline__ double2 operator-(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__host__ __device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__host__ __device__ __forceinline__ double2 cmul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
// acc + x*w as four fused multiply-adds, the SAMPLE as the broadcast operand: on sm_100 two FFMA2 (a scalar broadcast is a free
// operand modifier of the packed pipe, a half swap is not -- tools/ubench_fp32x2_mod.cu), with (-w.y, w.x) hoisted per tap
__device__ __forceinline__ float2 cmac(float2 acc, float2 x, float2 w) {
    acc = __ffma2_rn(make_float2(x.x, x.x), w, acc);
    return __ffma2_rn(make_float2(x.y, x.y), make_float2(-w.y, w.x), acc);
}
__device__ __forceinline__ double2 cmac(double2 acc, double2 x, double2 w) {
    return make_double2(fma(x.y, -w.y, fma(x.x, w.x, acc.x)), fma(x.y, w.x, fma(x.x, w.y, acc.y)));
}
// a * conj(b)
__host__ __device__ __forceinline__ float2 cmulc(float2 a, float2 b) { return make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); }
__host__ __device__ __forceinline__ double2 cmulc(double2 a, double2 b) { return make_double2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); }
__host__ __device__ __forceinline__ float2 cconj(float2 a) { return make_float2(a.x, -a.y); }
__host__ __device__ __forceinline__ double2 cconj(double2 a) { return make_double2(a.x, -a.y); }
__host__ __device__ __forceinline__ float2 cscale(float2 a, float s) { return make_float2(a.x * s, a.y * s); }
__host__ __device__ __forceinline__ double2 cscale(double2 a, double s) { return make_double2(a.x * s, a.y * s); }
__host__ __device__ __forceinline__ float cabs2(float2 a) { return a.x * a.x + a.y * a.y; }
__host__ __device__ __forceinline__ double cabs2(double2 a) { return a.x * a.x + a.y * a.y; }
// a / b  (plain textbook quotient; the oracle's double division differs only in rounding)
__host__ __device__ __forceinline__ float2 cdiv(float2 a, float2 b) {
    float d = b.x * b.x + b.y * b.y;
    return make_float2((a.x * b.x + a.y * b.y) / d, (a.y * b.x - a.x * b.y) / d);
}
__host__ __device__ __forceinline__ double2 cdiv(double2 a, double2 b) {
    double d = b.x * b.x + b.y * b.y;
    return make_double2((a.x * b.x + a.y * b.y) / d, (a.y * b.x - a.x * b.y) / d);
}
// multiply by -i (forward) / +i (inverse)
template <typename C> __device__ __forceinline__ C mul_mi(C a) { C r; r.x = a.y; r.y = -a.x; return r; }
template <typename C> __device__ __forceinline__ C mul_pi(C a) { C r; r.x = -a.y; r.y = a.x; return r; }

__device__ __forceinline__ double2 to_d(float2 a) { return make_double2((double)a.x, (double)a.y); }
__device__ __forceinline__ double2 to_d(double2 a) { return a; }
template <typename T> __device__ __forceinline__ cx<T> from_d(double2 a) { return mk<T>((T)a.x, (T)a.y); }

// ------------------------------------------------------------------ reductions
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// block-wide sum; `red` is >= 32 elements of shared scratch; result valid in every thread.
template <typename V> __device__ __forceinline__ V block_sum(V v, V* red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    V r = (lane < nw) ? red[lane] : V(0);
    r = warp_sum(r);
    return r;
}
// exclusive prefix sum of one int per thread over the block (blockDim.x a multiple of 32, <= 1024); `sh` >= 32 ints of
// shared scratch.  Two barriers inside; the result is valid in every thread.
__device__ __forceinline__ int block_exclusive_scan(int v, int* sh) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    __syncthreads();
    if (lane == 31) sh[w] = incl;
    __syncthreads();
    int base = 0;
    for (int k = 0; k < w; ++k) base += sh[k];
    return base + incl - v;
}
__device__ __forceinline__ int block_min(int v, int* red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_min(v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    int r = (lane < nw) ? red[lane] : 0x7fffffff;
    return warp_min(r);
}

// ------------------------------------------------------------------ packed-bit helpers
// 32 stream bits starting at absolute bit position `pos` (bits beyond `total` read as 0).
__device__ __forceinline__ uint32_t bits_get32(const uint32_t* __restrict__ w, int64_t pos, int64_t total) {
    if (pos >= total) return 0u;
    int64_t wi = pos >> 5;
    int sh = (int)(pos & 31);
    int64_t nwords = (total + 31) >> 5;
    uint32_t lo = w[wi];
    uint32_t hi = (sh != 0 && wi + 1 < nwords) ? w[wi + 1] : 0u;
    uint32_t v = __funnelshift_r(lo, hi, sh);
    int64_t rem = total - pos;
    if (rem < 32) v &= (1u << (int)rem) - 1u;
    return v;
}
// OR `n` (1..32) bits of v into a zero-initialised packed buffer at absolute bit position pos.
__device__ __forceinline__ void bits_put(uint32_t* w, int64_t pos, int n, uint32_t v) {
    if (n < 32) v &= (1u << n) - 1u;
    int64_t wi = pos >> 5;
    int sh = (int)(pos & 31);
    if (sh == 0 && n == 32) { w[wi] = v; return; }
    atomicOr(&w[wi], v << sh);
    if (sh + n > 32) atomicOr(&w[wi + 1], v >> (32 - sh));
}
// Word w of DeScrambler(s) for a word-aligned stream of frames of frame_bits >= 64 bits, from the raw words R = s word w and
// P = s word w - 1 (0 at w = 0): out[i] = s[i] ^ s[i-13] ^ s[i-14] on the 64-bit window (P : R).  Frames need not be word
// aligned: where a frame starts inside the window the bits below it are replaced by the initial register's history prev0
// (`DeScrambler.m:8-13` with the per-frame reset of `Main_model_Task_4.m:350-364`), and the word's bits before the boundary
// keep the previous frame's history.
__device__ __forceinline__ uint32_t descramble_word(uint32_t R, uint32_t P, int w, int frame_bits, uint32_t prev0) {
    auto window = [](unsigned long long x) { return (uint32_t)((x ^ (x << 13) ^ (x << 14)) >> 32); };
    const unsigned long long X = ((unsigned long long)R << 32) | P;
    uint32_t o = window(X);
    const int fl = (32 * w + 31) / frame_bits;                  // frame of the word's last bit
    const int t = fl * frame_bits - 32 * w;                     // its start relative to this word: (-frame_bits, 31]
    if (t > -14) {
        const int sh = 32 + t;                                  // window position of the frame's first bit, 19..63
        const unsigned long long keep = ~0ull << sh;
        const unsigned long long hist = sh >= 32 ? ((unsigned long long)prev0 << (sh - 32)) : ((unsigned long long)prev0 >> (32 - sh));
        const uint32_t of = window((X & keep) | (hist & ~keep));
        const uint32_t before = t > 0 ? ((1u << t) - 1u) : 0u;  // bits of this word that still belong to the previous frame
        o = (o & before) | (of & ~before);
    }
    return o;
}

// ------------------------------------------------------------------ constellation tables
struct ConstTable {
    int bps;
    double re[16], im[16];
};
ConstTable host_constellation(int id);  // api.cu

template <typename T> struct DevConst {
    int bps, n;
    T re[16], im[16];
};
template <typename T> inline DevConst<T> make_devconst(int id) {
    ConstTable c = host_constellation(id);
    DevConst<T> d;
    d.bps = c.bps;
    d.n = 1 << c.bps;
    for (int i = 0; i < 16; ++i) { d.re[i] = (T)c.re[i]; d.im[i] = (T)c.im[i]; }
    return d;
}
// min squared-Euclid index, strict '<' => first minimum, NaN never wins (`demapping.m:9-12`).
template <typename T> __device__ __forceinline__ int nearest_idx(const DevConst<T>& c, T x, T y, T* margin) {
    T best = CUDART_INF, second = CUDART_INF;
    int bi = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        if (i < c.n) {
            T dx = x - c.re[i], dy = y - c.im[i];
            T d = dx * dx + dy * dy;
            if (d < best) { second = best; best = d; bi = i; }
            else if (d < second) second = d;
        }
    }
    if (margin) *margin = second - best;
    return bi;
}

// ------------------------------------------------------------------ context
struct InterpPlan {       // device-resident spline/linear operator for a fixed knot set
    int n_knots;          // after edge extension
    int n_src;            // knot values supplied by the caller (Np)
    int ext_lo, ext_hi;   // 1 when an extrapolated knot is prepended / appended
    int nq;               // query points
    int hb;               // half bandwidth of the derivative operator
    int folded;           // 1: the edge extension is folded into the operator (it never reads knots 0 / n-1)
    double lo_den, lo_mul, hi_den, hi_mul;  // edge extension: slope denominators / distances
    void* band;           // (2hb+1) x n_knots real (T), tap-major so that threads (= knots) load coalesced
    void* qw;             // 4 x nq real (T) Hermite weights, one plane per weight
    int32_t* qk;          // nq interval index
};

struct BlobEntry { void* dev; size_t bytes; uint64_t check; };
#define OFDM_BLOB_CACHE_LIMIT 4096
#define OFDM_PLAN_CACHE_LIMIT 512

struct ofdm_ctx {
    int device = 0;
    int precision = OFDM_PREC_F32;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream[2] = {nullptr, nullptr};
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int sm_count = 148;
    int64_t launches = 0;
    std::string err;
    std::map<uint64_t, BlobEntry> blob_cache;      // small host config blobs mirrored on device (live generation)
    std::map<uint64_t, BlobEntry> blob_retired;    // previous generation: freed when the live one overflows again
    std::map<uint64_t, void*> twiddle_cache;       // key = N<<1 | prec (N a power of two <= 8192: bounded by construction)
    std::map<uint64_t, InterpPlan> plan_cache, plan_retired;
    std::vector<void*> owned;                      // freed at destroy
    void* scratch = nullptr;
    size_t scratch_bytes = 0;
    void* staging[2] = {nullptr, nullptr};         // device staging for the *_host chain
    size_t staging_bytes = 0;
    int64_t* host_counts_d = nullptr;              // {errors, bits, near} of the *_host chain (in `owned`)
};

int ctx_fail(ofdm_ctx* ctx, int code, const char* fmt, ...);
void* ctx_blob(ofdm_ctx* ctx, const void* host, size_t bytes);           // cached upload (by content hash)
cudaError_t ctx_upload(void* dev, const void* host, size_t bytes);       // pageable H2D, complete on return
void* ctx_scratch(ofdm_ctx* ctx, size_t bytes);                          // grow-only scratch
const void* ctx_twiddles(ofdm_ctx* ctx, int N);                          // W_N^k, k=0..N-1, ctx precision
const void* ctx_twiddles_prec(ofdm_ctx* ctx, int N, int precision);      // same table in a given precision
const InterpPlan* ctx_plan(ofdm_ctx* ctx, const int32_t* knots1, int n, int ext_to /*0=no ext*/,
                           const int32_t* queries1 /*NULL => 1..nq*/, int nq, int method);
uint64_t fnv1a(const void* p, size_t n, uint64_t h = 1469598103934665603ull);
// Opt-in to `bytes` of dynamic shared memory for kernel `func` on the current device.  The limit belongs to the device's copy
// of the kernel, not to a context, so contexts driven from several host threads (ofdm_group) share it: a plain
// cudaFuncSetAttribute by one thread could LOWER it between another thread's opt-in and launch.  This one only ever raises it,
// under a process-wide lock.
cudaError_t func_smem_optin(const void* func, int bytes);

#define CUDA_TRY(ctx, expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return ctx_fail(ctx, OFDM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
#define LAUNCH_CHECK(ctx)                                                                     \
    do {                                                                                      \
        (ctx)->launches++;                                                                    \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess)                                                                \
            return ctx_fail(ctx, OFDM_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
#define REQUIRE(ctx, cond, msg)                                                               \
    do {                                                                                      \
        if (!(cond)) return ctx_fail(ctx, OFDM_ERR_INVALID, "%s: %s", __func__, msg);         \
    } while (0)
// dispatch on the context's real type
#define DISPATCH_T(ctx, ...)                                                                  \
    do {                                                                                      \
        if ((ctx)->precision == OFDM_PREC_F64) { using T = double; __VA_ARGS__ }              \
        else { using T = float; __VA_ARGS__ }                                                 \
    } while (0)

static inline int ilog2(int n) { int l = 0; while ((1 << l) < n) ++l; return l; }
static inline bool is_pow2(int n) { return n > 0 && (n & (n - 1)) == 0; }
static inline int64_t cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }
