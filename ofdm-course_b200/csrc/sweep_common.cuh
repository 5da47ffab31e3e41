// The tile driver of the ofdm_sweep_* entry points: this rank's share of the streams walked in tiles that never straddle a
// point, one stream-ordered allocation for the temporaries of a tile, and the dense multipath response of a tap list.
#pragma once
#include <cmath>
#include <initializer_list>

#include "common.cuh"

// The payload of streams g .. g + n - 1 as ofdm_sweep_ber draws it (sweep.cu)
int ofdm_sweep_tile_payload(ofdm_ctx* ctx, const ofdm_link_params* lp, uint32_t* sbits, uint32_t* bits, int64_t n, int64_t words, uint64_t seed, int64_t g);
// Per stream of a tile of n: the SNR the channel reads and, when `fixed`, the STO and CFO (sweep_sync.cu)
void ofdm_sweep_fill(ofdm_ctx* ctx, int64_t n, double snr_db, int fixed, int32_t sto, double cfo, double* snr, int32_t* nsto, double* cfo_out);
// n streams of stream_bits bits, each the first bits of wpad padded words of `raw`, as one contiguous bitstream (sweep_sync.cu)
void ofdm_sweep_pack_bits(ofdm_ctx* ctx, const uint32_t* raw, int64_t n, int64_t wpad, int64_t stream_bits, uint32_t* out);

// Rank `rank` of `world` takes the contiguous share [first, first + count) of the n_points x per_point global streams
// g = point * per_point + j (ofdm_sweep_share).  tile = min(tile_streams > 0 ? tile_streams : tile_default, per_point).
struct SweepTiles {
    int64_t per_point, first = 0, count = 0, tile;
    SweepTiles(int64_t n_points, int64_t per_point_, int rank, int world, int64_t tile_streams, int64_t tile_default)
        : per_point(per_point_), tile(std::min<int64_t>(tile_streams > 0 ? tile_streams : tile_default, per_point_)) {
        ofdm_sweep_share(n_points * per_point, rank, world, &first, &count);
    }
    // body(point, first_in_point, g, n) for every tile of at most `tile` streams g .. g + n - 1 of one point, in order, until
    // it returns non-zero; returns that value (OFDM_OK when every tile ran)
    template <typename Body> int walk(Body&& body) const {
        for (int64_t g = first; g < first + count;) {
            const int64_t i = g / per_point, j0 = g - i * per_point;
            const int64_t n = std::min<int64_t>(std::min<int64_t>(tile, first + count - g), per_point - j0);
            if (const int rc = body(i, j0, g, n)) return rc;
            g += n;
        }
        return OFDM_OK;
    }
};

// One cudaMallocAsync on the context's stream carved into blocks of the given byte sizes, each padded to 256 bytes; freed
// with cudaFreeAsync when the object goes out of scope, after everything enqueued on the stream before.
class SweepScratch {
public:
    explicit SweepScratch(ofdm_ctx* ctx) : ctx_(ctx) {}
    SweepScratch(const SweepScratch&) = delete;
    SweepScratch& operator=(const SweepScratch&) = delete;
    ~SweepScratch() { if (base_) cudaFreeAsync(base_, ctx_->stream); }
    cudaError_t alloc(std::initializer_list<size_t> bytes) {
        size_t total = 0;
        for (size_t b : bytes) { off_.push_back(total); total += (b + 255) / 256 * 256; }
        return cudaMallocAsync((void**)&base_, total, ctx_->stream);
    }
    template <typename T> T* get(size_t block) const { return (T*)(base_ + off_[block]); }
    // the closing check of a sweep: a launch error not reported yet fails the call with "<what>: <CUDA error>"
    int finish(int rc, const char* what) const {
        const cudaError_t e = cudaGetLastError();
        if (rc == OFDM_OK && e != cudaSuccess) rc = ctx_fail(ctx_, OFDM_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
        return rc;
    }

private:
    ofdm_ctx* ctx_;
    unsigned char* base_ = nullptr;
    std::vector<size_t> off_;
};

// The dense impulse response h(1:D) of a (delay, amplitude) tap list, D = largest delay + 1 (`get_MP_channel_resp.m:2-19`:
// later rows overwrite earlier ones).  False when a delay is not an integer in [0, max_delay).
static inline bool sweep_dense_taps(const double* taps, int n_taps, int max_delay, std::vector<double>& h) {
    int D = 0;
    for (int k = 0; k < n_taps; ++k) {
        const double d = taps[2 * k];
        if (!(d >= 0 && d < max_delay && d == floor(d))) return false;
        D = std::max(D, (int)d + 1);
    }
    h.assign(D, 0.0);
    for (int k = 0; k < n_taps; ++k) h[(int)taps[2 * k]] = taps[2 * k + 1];
    return true;
}
