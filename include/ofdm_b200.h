/*
 * libofdm_b200 -- C ABI of the B200-native batched OFDM link chain.
 *
 * The reference (ladnlav/OFDM-course, plain MATLAB) exposes no FFI: its boundary is the set of
 * MATLAB function signatures in `Task 5/<name>.m` (plus `Task 4/fine_sync.m` and the v1 mapper in
 * `Task 1/OFDM_map_carriers.m`).  Every entry point below replaces exactly one of those functions
 * (cited as path:line under /root/reference) and is what the MEX gateway `mex/ofdm_mex.c`, the
 * ctypes binding `ofdm-course_b200/_cabi.py`, or any other FFI binds.  See INTEGRATION.md.
 *
 * Conventions
 *   - Batched: the leading dimension B runs over independent serial streams (the reference
 *     processes one stream per script run).  Within a stream the layout is MATLAB's column-major
 *     matrix, i.e. symbol-major: grid[b][s][k], k = 0..Nfft-1.
 *   - "dev" pointers are device memory of the context's GPU; "host" pointers are small shared
 *     configuration (index lists, pilot values, taps, the 15-cell register) that the library
 *     caches on the device.  Carrier / pilot / tap index lists are **1-based**, as in MATLAB.
 *   - Complex samples are interleaved (re,im) pairs of the context's real type: float
 *     (OFDM_PREC_F32) or double (OFDM_PREC_F64, the closer-comparison mode).
 *   - Bit vectors are packed bitstreams, LSB-first inside little-endian 32-bit words: stream bit i
 *     is `(w[i>>5] >> (i&31)) & 1` (== numpy.packbits(..., bitorder='little')).  Buffers hold
 *     OFDM_BIT_WORDS(n) words.
 *   - Every function returns OFDM_OK (0) or a negative status; `ofdm_last_error` gives the text.
 *     Nothing throws across the ABI.  All work is enqueued on the context's stream; results are
 *     complete after `ofdm_sync` (or any stream synchronisation by the caller).
 *   - There is NO CPU fallback: a context cannot be created without an sm_100 device.
 */
#ifndef OFDM_B200_H
#define OFDM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFDM_API __attribute__((visibility("default")))

#define OFDM_OK 0
#define OFDM_ERR_INVALID (-1)   /* bad argument */
#define OFDM_ERR_CUDA (-2)      /* CUDA runtime failure (text in ofdm_last_error) */
#define OFDM_ERR_NODEVICE (-3)  /* no sm_100 device: there is no CPU fallback */
#define OFDM_ERR_UNSUPPORTED (-4)

#define OFDM_PREC_F32 0
#define OFDM_PREC_F64 1

/* constellation ids, `Task 5/constellation_func.m:5-19` */
#define OFDM_BPSK 1
#define OFDM_QPSK 2
#define OFDM_8PSK 3
#define OFDM_16QAM 4

#define OFDM_INTERP_LINEAR 0
#define OFDM_INTERP_SPLINE 1

#define OFDM_BIT_WORDS(nbits) (((nbits) + 31) / 32)

typedef struct ofdm_ctx ofdm_ctx;

/* ---- context, memory, stream ------------------------------------------------------------ */
OFDM_API int ofdm_ctx_create(ofdm_ctx** out, int device, int precision);
OFDM_API void ofdm_ctx_destroy(ofdm_ctx* ctx);
OFDM_API const char* ofdm_last_error(const ofdm_ctx* ctx);
OFDM_API int ofdm_ctx_set_stream(ofdm_ctx* ctx, void* cuda_stream); /* cudaStream_t; NULL = own stream; (void*)1 = cudaStreamLegacy */
OFDM_API int ofdm_sync(ofdm_ctx* ctx);
OFDM_API int ofdm_precision(const ofdm_ctx* ctx);
OFDM_API int ofdm_malloc(ofdm_ctx* ctx, void** dev, size_t bytes);
OFDM_API int ofdm_free(ofdm_ctx* ctx, void* dev);
OFDM_API int ofdm_memset(ofdm_ctx* ctx, void* dev, int value, size_t bytes);
OFDM_API int ofdm_h2d(ofdm_ctx* ctx, void* dev, const void* host, size_t bytes);
OFDM_API int ofdm_d2h(ofdm_ctx* ctx, void* host, const void* dev, size_t bytes);
OFDM_API int ofdm_host_alloc(void** host, size_t bytes); /* pinned */
OFDM_API int ofdm_host_free(void* host);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
OFDM_API int64_t ofdm_launch_count(const ofdm_ctx* ctx);
OFDM_API const char* ofdm_version(void);

/* ---- a1/a2  Scrambler / DeScrambler  (`Task 5/Scrambler.m:1-28`, `DeScrambler.m:1-28`) --- */
/* n_frames frames of frame_bits bits, contiguous in one bitstream; every frame starts from the
 * same 15-cell register `reg0_host` (per-frame reset, `Task 4/Main_model_Task_4.m:43-58`).
 * final_regs_dev (optional) receives n_frames x 15 bytes: the register after each frame. */
OFDM_API int ofdm_scramble(ofdm_ctx*, const uint32_t* in_dev, uint32_t* out_dev, int64_t n_frames,
                           int64_t frame_bits, const uint8_t* reg0_host, uint8_t* final_regs_dev);
OFDM_API int ofdm_descramble(ofdm_ctx*, const uint32_t* in_dev, uint32_t* out_dev, int64_t n_frames,
                             int64_t frame_bits, const uint8_t* reg0_host, uint8_t* final_regs_dev);

/* ---- a3  constellation_func  (`Task 5/constellation_func.m:4-29`) ------------------------ */
/* table_host: 2*2^bps doubles (re,im); returns bits per symbol through bps. */
OFDM_API int ofdm_constellation(int constellation, double* table_host, int* bps);

/* ---- a4/a5  mapping / demapping  (`Task 5/mapping.m:1-25`, `demapping.m:1-25`) ----------- */
/* n_bits bits -> ceil(n_bits/bps) symbols (zero padded); *pad = -1 when nothing was padded. */
OFDM_API int ofdm_map(ofdm_ctx*, const uint32_t* bits_dev, int64_t n_bits, int constellation,
                      void* iq_dev, int* pad);
/* n_sym symbols -> n_sym*bps bits (caller drops the trailing `pad` bits exactly as demapping.m:21-23).
 * near_dev (optional, one int64): incremented for every symbol whose two smallest squared
 * distances differ by less than `near_eps` (a decision within epsilon of a boundary). */
OFDM_API int ofdm_demap(ofdm_ctx*, const void* iq_dev, int64_t n_sym, int constellation,
                        uint32_t* bits_dev, double near_eps, int64_t* near_dev);

/* ---- a6  OFDM_map_carriers  (`Task 5/OFDM_map_carriers.m:2-8`; v1 `Task 1/...:2-12`) ------ */
/* qam_dev: B x (Nd*S); grid_dev: B x S x Nfft.  pilot_vals_host: Np*S complex doubles
 * (column-major Np x S) when pilot_mode = 0, one complex double (scalar broadcast) when 1,
 * one real amplitude expanded to alternating +a, a*exp(i*pi) (v1) when 2. */
OFDM_API int ofdm_map_carriers(ofdm_ctx*, const void* qam_dev, int64_t B, int S, int Nfft,
                               const int32_t* data_carriers_host, int Nd,
                               const int32_t* pilot_carriers_host, int Np,
                               const double* pilot_vals_host, int pilot_mode, void* grid_dev);

/* ---- a7/a8/a9  OFDM_modulator / OFDM_demodulator / get_payload ---------------------------- */
/* (`Task 5/OFDM_modulator.m:2-10`, `OFDM_demodulator.m:2-9`, `get_payload.m:2-4`) */
OFDM_API int ofdm_modulate(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft, int Tg,
                           void* time_dev /* B x S x (Nfft+Tg) */);
OFDM_API int ofdm_demodulate(ofdm_ctx*, const void* time_dev, int64_t B, int S, int Nfft, int Tg,
                             void* grid_dev /* B x S x Nfft */);
OFDM_API int ofdm_get_payload(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft,
                              const int32_t* data_carriers_host, int Nd, void* iq_dev /* B x S x Nd */);
/* plain batched FFT (inverse != 0: MATLAB ifft with 1/N) over n_batch contiguous length-N vectors */
OFDM_API int ofdm_fft(ofdm_ctx*, const void* in_dev, void* out_dev, int64_t n_batch, int N, int inverse);

/* ---- a10-a13  add_STO / add_CFO / Noise / get_MP_channel_resp + conv ---------------------- */
/* (`Task 5/add_STO.m:1-10`, `add_CFO.m:1-8`, `Noise.m:1-12`, `get_MP_channel_resp.m:2-19`,
 *  conv + truncate `Task 5/Main_model_Task_5.m:126-127`).  Streams are B x L. */
OFDM_API int ofdm_add_sto(ofdm_ctx*, const void* in_dev, int64_t B, int64_t L, const int32_t* nsto_dev,
                          void* out_dev);
OFDM_API int ofdm_add_cfo(ofdm_ctx*, const void* in_dev, int64_t B, int64_t L, const double* cfo_dev,
                          int Nfft, void* out_dev);
/* normals_dev: B x 2 x L unit normals of the context's real type (real block, then imaginary block,
 * the order of the two normrnd calls) or NULL -> Philox4x32-10 keyed by (seed, first_stream_id + b).
 * snr_db_dev: B doubles.  nvar_dev (optional): B doubles = sqrt(NoisePower). */
OFDM_API int ofdm_add_noise(ofdm_ctx*, const void* in_dev, int64_t B, int64_t L, const double* snr_db_dev,
                            const void* normals_dev, uint64_t seed, int64_t first_stream_id,
                            void* out_dev, double* nvar_dev);
/* taps_host: K x 2 doubles (delay, amplitude) row-major.  h_host: *h_len doubles out (max_delay+1);
 * H_dev (optional): Nfft complex = fft(h, Nfft). */
OFDM_API int ofdm_mp_channel_resp(ofdm_ctx*, const double* taps_host, int K, int Nfft, double* h_host,
                                  int h_cap, int* h_len, void* H_dev);
/* h_dev: complex FIR of length D, one per stream (h_per_stream != 0) or shared. */
OFDM_API int ofdm_apply_fir(ofdm_ctx*, const void* in_dev, int64_t B, int64_t L, const void* h_dev, int D,
                            int h_per_stream, void* out_dev);

/* Static tapped-delay-line fading channel standing in for `lteFadingChannel` as used by `Task 5/Task5_part2.m:27-34,
 * 152-154` (DopplerFreq 0, one realisation per Monte-Carlo run): profile 0 EPA, 1 EVA, 2 ETU (3GPP TS 36.101 B.2.1),
 * Rayleigh tap gains from Philox keyed by (seed, first_stream_id + b), fractional delays by a windowed-sinc
 * interpolator with a lead of 7 samples.  LTE Toolbox internals are not public: draws differ from MATLAB's.
 * ofdm_tdl_info: n_paths (= dominant_taps of the MP/OMP calls), h_len, path delays in samples (<= 9 doubles).
 * ofdm_tdl_channel: h_dev B x h_len complex impulse responses (feed to ofdm_apply_fir, h_per_stream = 1),
 * gains_dev optional B x n_paths. */
OFDM_API int ofdm_tdl_info(int profile, double fs_hz, int* n_paths, int* h_len, double* delays_samples);
OFDM_API int ofdm_tdl_channel(ofdm_ctx*, int profile, double fs_hz, int64_t B, uint64_t seed, int64_t first_stream_id,
                              int h_len, void* h_dev, void* gains_dev);
/* (H - Hest)(H - Hest)' / n per stream (`Task 5/Task5_part2.m:200-203`): out_dev B doubles. */
OFDM_API int ofdm_mse(ofdm_ctx*, const void* a_dev, int64_t a_stride, const void* b_dev, int64_t b_stride, int64_t B,
                      int n, double* out_dev);

/* ---- a14-a16  AutoCorrFunction / remove_IFO / fine_sync ----------------------------------- */
/* (`Task 5/AutoCorrFunction.m:1-28`) autocorr_dev optional: B x (L-W-Nfft) complex.
 * tg_pos_dev: B int32 (1-based, 65 on detector failure), freq_off_dev: B doubles,
 * fail_dev (optional): B int32, 1 where the fallback 65 was taken. */
OFDM_API int ofdm_cp_autocorr(ofdm_ctx*, const void* rx_dev, int64_t B, int64_t L, int W, int Nfft,
                              void* autocorr_dev, int32_t* tg_pos_dev, double* freq_off_dev, int32_t* fail_dev);
/* (`Task 5/remove_IFO.m:1-11`) ifo_dev: B int32; -1 where no bin exceeds 0.77 (MATLAB errors there;
 * the stream is then passed through unchanged). */
OFDM_API int ofdm_remove_ifo(ofdm_ctx*, const void* rx_dev, int64_t B, int64_t L, int Nfft, void* out_dev,
                             int32_t* ifo_dev);
/* (`Task 4/fine_sync.m:1-60`) grids are B x S x Nfft; pilot_vals_host Np x S complex doubles.
 * tau_dev / phase_dev (optional): B doubles. */
OFDM_API int ofdm_fine_sync(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft,
                            const int32_t* pilot_carriers_host, int Np, const double* pilot_vals_host,
                            int time_desync, int freq_desync, void* out_dev, double* tau_dev, double* phase_dev);

/* ---- a17-a21  estimate_channel / LS_CE / MMSE_CE / interpolate / equalize_signal ---------- */
/* (`Task 5/estimate_channel.m:1-10`) H_dev: B x Nq over the query carriers; Hp_dev optional B x Np. */
OFDM_API int ofdm_estimate_channel(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft,
                                   const int32_t* all_carriers_host, int Nq,
                                   const int32_t* pilot_carriers_host, int Np,
                                   const double* pilot_vals_host, void* H_dev, void* Hp_dev);
/* (`Task 5/LS_CE.m:1-34`) first symbol only; H_dev: B x N_carrier. */
OFDM_API int ofdm_ls_ce(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft,
                        const int32_t* pilot_loc_host, int Np, const double* pilot_vals_host,
                        int N_carrier, void* H_dev);
/* (`Task 5/MMSE_CE.m:1-39`) h_dev: B x h_len complex channel impulse responses; snr_db_dev: B doubles. */
OFDM_API int ofdm_mmse_ce(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft,
                          const int32_t* pilot_loc_host, int Np, const double* pilot_vals_host,
                          int N_carrier, const void* h_dev, int h_len, const double* snr_db_dev, void* H_dev);
/* MMSE_CE for a batch that shares its channel statistics (one Monte-Carlo point, `Task 5/Task5_part2.m:176-177`): ONE
 * impulse response h_dev (h_len complex, gives tau_rms) and ONE SNR for all B streams.  W = I - Rpp^{-1}/snr is built once
 * and applied to every stream as a complex matrix product on the tensor cores (TF32 two-term split, FP32 accuracy). */
OFDM_API int ofdm_mmse_ce_shared(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft,
                                 const int32_t* pilot_loc_host, int Np, const double* pilot_vals_host,
                                 int N_carrier, const void* h_dev, int h_len, double snr_db, void* H_dev);
/* (`Task 5/interpolate.m:1-24`) Hp_dev: B x Np -> H_dev: B x N. */
OFDM_API int ofdm_interpolate(ofdm_ctx*, const void* Hp_dev, int64_t B, const int32_t* pilot_loc_host, int Np,
                              int N, int method, void* H_dev);
/* (`Task 5/equalize_signal.m:1-8`) H_dev: B x h_stride (>= N_carrier); rows > N_carrier become 0. */
OFDM_API int ofdm_equalize(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft, const void* H_dev,
                           int h_stride, int N_carrier, void* out_dev);

/* Measurement vector of the sparse estimators, `Y = RX(pilotCarriers,1)./pilotValues(:,1)`
 * (`Task 5/Main_model_Task_5.m:191`, `Task5_part2.m:190`): y_dev B x Np from grid_dev B x S x Nfft. */
OFDM_API int ofdm_pilot_ls(ofdm_ctx*, const void* grid_dev, int64_t B, int S, int Nfft, const int32_t* pilot_loc_host,
                           int Np, const double* Xp_host, void* y_dev);

/* ---- a22/a23  OMP_estimate / MP_estimate  (`Task 5/OMP_estimate.m:2-37`, `MP_estimate.m:2-34`) */
/* y_dev: B x Np.  Dictionary: either dense `A_dev` (Np x Ldict, column-major as MATLAB stores
 * sensing_matrix, shared by the batch) or, when A_dev == NULL, the partial-DFT descriptor
 * A(i,l) = exp(-2*pi*1j*(pilot_loc[i]-1)*(l-1)/Nfft) (`Task 5/Main_model_Task_5.m:182-190`), for which
 * the correlation A^H r runs as a scatter + inverse FFT.  Outputs: H_dev B x Nfft, h_dev B x Nfft,
 * index_dev B x K int32 (1-based, 0 = unused slot), iters_dev B int32 (columns selected). */
OFDM_API int ofdm_omp(ofdm_ctx*, const void* y_dev, int64_t B, int Np, const void* A_dev, int Ldict,
                      const int32_t* pilot_loc_host, int Nfft, int K, void* H_dev, void* h_dev,
                      int32_t* index_dev, int32_t* iters_dev);
/* Same, and near_ties_dev (optional, B int32) receives per frame the number of iterations whose two largest |A^H r|^2
 * differ by less than tie_eps (relative): the tap ORDER of such a frame may differ from a float64 evaluation.
 * Partial-DFT dictionaries (the descriptor, or a dense matrix recognised as one) run as Batch-OMP -- one FFT per frame
 * and the Toeplitz Gram vector; unstructured dense dictionaries in large batches run their correlations on tcgen05. */
OFDM_API int ofdm_omp_ex(ofdm_ctx*, const void* y_dev, int64_t B, int Np, const void* A_dev, int Ldict,
                         const int32_t* pilot_loc_host, int Nfft, int K, void* H_dev, void* h_dev,
                         int32_t* index_dev, int32_t* iters_dev, int32_t* near_ties_dev, double tie_eps);
OFDM_API int ofdm_mp(ofdm_ctx*, const void* y_dev, int64_t B, int Np, const void* A_dev, int Ldict,
                     const int32_t* pilot_loc_host, int Nfft, int K, void* H_dev, void* h_dev,
                     int32_t* index_dev);

/* ---- a24/a25  BER_func / MER_func  (`Task 5/BER_func.m:1-7`, `MER_func.m:1-26`) ----------- */
/* counts_dev: 2 int64 {errors, bits}, accumulated (+=) so sweeps can reuse one counter. */
OFDM_API int ofdm_ber_count(ofdm_ctx*, const uint32_t* tx_bits_dev, const uint32_t* rx_bits_dev,
                            int64_t n_bits, int64_t* counts_dev);
/* sums_dev: 2 doubles {sum |ideal|^2, sum |ideal-rx|^2}, accumulated (+=). */
OFDM_API int ofdm_mer(ofdm_ctx*, const void* iq_dev, int64_t n_sym, int constellation, double* sums_dev);

/* ---- PAPR / CCDF  (`Task 5/calculatePAPR.m:2-11`, `calculate_window_PAPR.m:2-15`, `calculateCCDF.m:2-6`) ---- */
/* x_dev: B x L streams.  papr_db_dev: B doubles = 10*log10(max|x|^2 / mean|x|^2). */
OFDM_API int ofdm_papr(ofdm_ctx*, const void* x_dev, int64_t B, int64_t L, double* papr_db_dev);
/* paprs_dev: B x (L - Nfft + 1) reals of the context's type: PAPR of every Nfft-sample window, O(L) per stream. */
OFDM_API int ofdm_window_papr(ofdm_ctx*, const void* x_dev, int64_t B, int64_t L, int Nfft, void* paprs_dev);
/* values_dev: n reals.  x_dev / ccdf_dev: capacity n + 1 reals; *n_out_dev entries are written:
 * MATLAB's ecdf support points (the minimum twice) and 1 - F at them. */
OFDM_API int ofdm_ccdf(ofdm_ctx*, const void* values_dev, int64_t n, void* x_dev, void* ccdf_dev, int64_t* n_out_dev);

/* ---- fused chains (the hot path) ----------------------------------------------------------- */
typedef struct ofdm_link_params {
    int32_t Nfft, Tg, N_carrier, S, SpF; /* S symbols per stream, SpF symbols per scrambler frame */
    int32_t constellation;
    int32_t Nd, Np;
    const int32_t* data_carriers_host;   /* Nd, 1-based */
    const int32_t* pilot_carriers_host;  /* Np, 1-based */
    const double* pilot_vals_host;       /* Np x S complex doubles, column-major */
    const uint8_t* reg0_host;            /* 15 */
    int32_t scramble;                    /* 0: skip Scrambler/DeScrambler (as `Task5_part2.m:99-115`) */
} ofdm_link_params;

/* TX: bits -> Scrambler (per-frame reset) -> mapping -> OFDM_map_carriers -> OFDM_modulator.
 * bits_dev: B streams x stream_bits (contiguous bitstream); time_dev: B x S x (Nfft+Tg).
 * (`Task 5/Main_model_Task_5.m:53-85`) */
OFDM_API int ofdm_tx_chain(ofdm_ctx*, const ofdm_link_params*, const uint32_t* bits_dev, int64_t B, void* time_dev);
/* Same, and also hands out sum |x|^2 of every stream (B doubles, cyclic prefixes included): the stream power `Noise.m:3`
 * measures, accumulated while the samples are still in registers so that ofdm_channel_t5_p need not re-read the signal. */
OFDM_API int ofdm_tx_chain_p(ofdm_ctx*, const ofdm_link_params*, const uint32_t* bits_dev, int64_t B, void* time_dev,
                             double* power_sum_dev);
/* Task-5 channel: AWGN (Philox or imported) then static multipath FIR
 * (`Task 5/Main_model_Task_5.m:108,123-127`); snr_db_dev may be NULL (no noise); h_dev NULL (no FIR). */
OFDM_API int ofdm_channel_t5(ofdm_ctx*, const void* tx_dev, int64_t B, int64_t L, const double* snr_db_dev,
                             const void* normals_dev, uint64_t seed, int64_t first_stream_id,
                             const void* h_dev, int D, void* rx_dev);
/* Same with the stream powers supplied (power_sum_dev: B doubles = sum |tx|^2 per stream, e.g. from ofdm_tx_chain_p);
 * NULL makes it measure them itself, which is what ofdm_channel_t5 does (`Task 5/Noise.m:3-5`). */
OFDM_API int ofdm_channel_t5_p(ofdm_ctx*, const void* tx_dev, int64_t B, int64_t L, const double* snr_db_dev,
                               const double* power_sum_dev, const void* normals_dev, uint64_t seed, int64_t first_stream_id,
                               const void* h_dev, int D, void* rx_dev);
/* Task-4 channel in one pass (`Task 4/Main_model_Task_4.m:95,103,110,263-264`): Noise -> add_STO(nsto) -> add_CFO(cfo) ->
 * multipath FIR; bit-identical to ofdm_add_noise -> ofdm_add_sto -> ofdm_add_cfo -> ofdm_apply_fir on the same arguments
 * (nsto_dev B int32 and cfo_dev B doubles as those calls take them; power_sum_dev may be NULL; h_dev D <= 1024 samples,
 * a single 1 for "no multipath"). */
OFDM_API int ofdm_channel_t4_p(ofdm_ctx*, const void* tx_dev, int64_t B, int64_t L, const double* snr_db_dev,
                               const double* power_sum_dev, const void* normals_dev, uint64_t seed, int64_t first_stream_id,
                               const int32_t* nsto_dev, const double* cfo_dev, int Nfft, const void* h_dev, int D, void* rx_dev);
/* M1 RX chain: OFDM_demodulator -> LS_CE -> equalize_signal -> get_payload -> demapping ->
 * DeScrambler -> BER count, one pass over the stream (`Task 5/Task5_part2.m:169-174,269-303`).
 * rx_dev B x S x (Nfft+Tg); tx_bits_dev reference bits (B x stream_bits); outputs (each optional):
 * out_bits_dev decided bits, H_dev B x N_carrier, counts_dev {errors, bits, near_boundary} int64 +=,
 * err_per_stream_dev B int32. */
OFDM_API int ofdm_rx_chain_t5(ofdm_ctx*, const ofdm_link_params*, const void* rx_dev, int64_t B,
                              const uint32_t* tx_bits_dev, uint32_t* out_bits_dev, void* H_dev,
                              int64_t* counts_dev, int32_t* err_per_stream_dev, double near_eps);
/* Same chain from HOST buffers (pinned or pageable), chunked and double-buffered over copy/compute
 * streams: the call a MATLAB/MEX user makes.  counts_host: 3 int64 (overwritten). */
OFDM_API int ofdm_rx_chain_t5_host(ofdm_ctx*, const ofdm_link_params*, const void* rx_host, int64_t B,
                                   const uint32_t* tx_bits_host, uint32_t* out_bits_host, void* H_host,
                                   int64_t* counts_host, int64_t chunk_streams);
/* Same with the near-boundary counter switched on: counts_host[2] = symbols whose two smallest squared distances to the
 * constellation differ by less than near_eps (the "within epsilon of a decision boundary" count of the parity contract). */
OFDM_API int ofdm_rx_chain_t5_host_eps(ofdm_ctx*, const ofdm_link_params*, const void* rx_host, int64_t B,
                                       const uint32_t* tx_bits_host, uint32_t* out_bits_host, void* H_host,
                                       int64_t* counts_host, int64_t chunk_streams, double near_eps);

/* M2 RX chain, fused (FP32 contexts): AutoCorrFunction -> add_STO x2 -> add_CFO -> remove_IFO -> OFDM_demodulator ->
 * fine_sync -> estimate_channel -> equalize_signal -> get_payload -> demapping -> DeScrambler -> BER count
 * (`Task 4/Main_model_Task_4.m:277-366`), one pass for the autocorrelation plus one persistent kernel.
 * rx_dev B x S x (Nfft+Tg).  Optional outputs: out_bits_dev, counts_dev {errors, bits, near} += , and the
 * per-stream estimates tg_dev (int32), fo_dev (double), ifo_dev (int32, -1 = no bin above 0.77), tau_dev,
 * phase_dev (double), H_dev (B x N_carrier).  A data carrier past N_carrier is decided from 0 (equalize_signal.m zeroes it);
 * with mp_desync = 0 such a layout returns OFDM_ERR_UNSUPPORTED, since the chain keeps only the N_carrier first bins. */
OFDM_API int ofdm_rx_chain_t4(ofdm_ctx*, const ofdm_link_params*, const void* rx_dev, int64_t B, int time_desync,
                              int freq_desync, int mp_desync, const uint32_t* tx_bits_dev, uint32_t* out_bits_dev,
                              int64_t* counts_dev, int32_t* tg_dev, double* fo_dev, int32_t* ifo_dev, double* tau_dev,
                              double* phase_dev, void* H_dev, double near_eps);
/* Same, and fail_dev (optional, B int32) receives 1 for every stream whose guard-interval detector found fewer than two
 * runs and fell back to TgPosition = 65 (`AutoCorrFunction.m:21-24`) -- the detector-failure count reported beside BER. */
OFDM_API int ofdm_rx_chain_t4_ex(ofdm_ctx*, const ofdm_link_params*, const void* rx_dev, int64_t B, int time_desync,
                                 int freq_desync, int mp_desync, const uint32_t* tx_bits_dev, uint32_t* out_bits_dev,
                                 int64_t* counts_dev, int32_t* tg_dev, double* fo_dev, int32_t* ifo_dev, double* tau_dev,
                                 double* phase_dev, void* H_dev, double near_eps, int32_t* fail_dev);

/* ---- Monte-Carlo BER-vs-SNR sweep (the script loops) ------------------------------------------ */
/* Replaces the SNR loop `Task 5/Main_model_Task_5.m:303-346` (chain OFDM_SWEEP_TASK5: TX chain -> Noise -> multipath -> M1
 * RX chain; the BER half of the Task-5 loop, ofdm_sweep_mse below runs its channel-estimation half; Task 3's loop, which has
 * no channel estimate, is ofdm_sweep_mer) and the impaired channel of
 * `Task 4/Main_model_Task_4.m:95-110,252-264,277-366` swept over SNR (chain OFDM_SWEEP_TASK4: TX chain -> Noise ->
 * add_STO -> add_CFO -> multipath -> M2 RX chain with AutoCorrFunction / remove_IFO / fine_sync / estimate_channel).
 * Streams are numbered globally, g = snr_index * streams_per_point + j; payload bits, noise, STO and CFO draws are
 * Philox streams keyed by (seed, g), so the integer counters are identical for every (rank, world, tile) split.
 * The payload is drawn in the scrambled domain: the Philox words of ofdm_payload_bits are the scrambled frames s and the
 * payload is p = DeScrambler(s) (uniform, and Scrambler(p) = s exactly), so the transmitter maps s without scrambling.
 * One call processes the rank-th of `world` equal contiguous shares of the global stream range (ofdm_sweep_share)
 * and ADDS into counts_dev: n_snr x 4 int64, row i = {bit errors, bits, symbols within near_eps of a decision
 * boundary, guard-interval detector failures (Task-4 chain)}.  The caller sums the rows of all ranks -- the path's
 * only collective, one int64 all-reduce.  Everything is enqueued on the context's stream. */
#define OFDM_SWEEP_TASK5 0
#define OFDM_SWEEP_TASK4 1
typedef struct ofdm_sweep_params {
    int32_t chain;               /* OFDM_SWEEP_TASK5 / OFDM_SWEEP_TASK4 */
    int32_t n_snr;
    const double* snr_db_host;   /* n_snr SNR points in dB */
    int64_t streams_per_point;
    int64_t tile_streams;        /* streams per work item; 0 = 8192 (two signal buffers of tile x stream bytes are allocated) */
    int32_t rank, world;         /* share of the global stream range this call processes */
    uint64_t seed;
    const double* taps_host;     /* n_taps x 2 doubles (delay, amplitude), row-major; n_taps = 0: no multipath */
    int32_t n_taps;
    double near_eps;             /* 0 = near-boundary counter off */
    int32_t sto_max;             /* Task-4 chain: Time_Delay ~ U{0..sto_max} (`Main_model_Task_4.m:101`: Nfft + T_Guard) */
    int32_t cfo_int_max;         /* Task-4 chain: Freq_Shift = U{0..cfo_int_max} + U(-0.5, 0.5) (`:108`: 30) */
} ofdm_sweep_params;
OFDM_API int ofdm_sweep_ber(ofdm_ctx*, const ofdm_link_params*, const ofdm_sweep_params*, int64_t* counts_dev);
/* Task-5 channel-estimation study over SNR (`Task 5/Main_model_Task_5.m:303-346`, MSE as `:195-205`): per stream Noise ->
 * multipath -> OFDM_demodulator -> LS_CE / MMSE_CE (h = ifft(H_LS), `:179`) / MP_estimate / OMP_estimate on the partial-DFT
 * dictionary of Ldict columns (`:182-190`, Ldict >= Np), and (H - Hest)(H - Hest)'/N_carrier against the true response
 * fft(h, Nfft)(1:N_carrier).  Uses chain (must be OFDM_SWEEP_TASK5), n_snr, snr_db_host, streams_per_point, tile_streams,
 * rank, world, seed, taps_host / n_taps (required, n_taps <= 32; K = n_taps dominant taps) and near_eps (OMP's tie_eps);
 * sto_max and cfo_int_max are ignored.  Share rule and stream numbering are those of ofdm_sweep_ber.  Nd == 0 transmits the
 * pilot-only stream (`:24-33`, the same for every g); Nd >= 1 the stream ofdm_sweep_ber transmits for g.  N_carrier must
 * be a power of two and the pilots lie in 1..N_carrier.
 * mse_dev: n_snr x 4 x streams_per_point doubles, [i][e][j] with e = LS, MMSE, MP, OMP; only this call's share is written.
 * counts_dev: n_snr x 2 int64 += {streams processed, OMP frames with a near-tie}.  The per-stream values do not depend on
 * the rank count or the tile size; the caller sums the arrays of all ranks (each cell is written by one rank). */
OFDM_API int ofdm_sweep_mse(ofdm_ctx*, const ofdm_link_params*, const ofdm_sweep_params*, int Ldict, double* mse_dev,
                            int64_t* counts_dev);
/* Task-5 part-2 pilot-density study (`Task 5/Task5_part2.m:46-321`): n_points pilot layouts x mc_runs static fading runs x
 * the LS / MMSE / MP / OMP estimators; for every cell the NMSE of the estimate (`:200-203`) and the bit errors after equalising
 * with it (`:269-303`).  From `base` the call reads Nfft, Tg, N_carrier, S, SpF and the constellation only; the data carriers
 * of a point are the complement of its pilots in 1..N_carrier, scrambling is off (`:99-115`).  Keys, those of the composed
 * Python driver part2.run_point: point k transmits the first S * Nd_k * bps payload bits through ofdm_tx_chain, gets AWGN
 * once (ofdm_add_noise, first_stream_id k), run r fades with ofdm_tdl_channel(first_stream_id k * 1,000,003 + r); MMSE gets
 * the true impulse response zero-padded to N_carrier, MP / OMP the partial-DFT dictionary of ldict_host[k] columns with
 * K = n_paths of the profile.  Work item g = k * mc_runs + r; the call processes the share ofdm_sweep_share(n_points *
 * mc_runs, rank, world) gives, in tiles of tile_runs runs (0 = 4096) that never straddle a point. */
typedef struct ofdm_part2_params {
    int32_t n_points;
    const int32_t* pilot_offsets_host;  /* n_points + 1, from 0: point k's pilots are pilot_carriers_host[off[k] .. off[k+1]) */
    const int32_t* pilot_carriers_host; /* 1-based, strictly increasing within 1..N_carrier per point, >= 2 per point */
    const int32_t* ldict_host;          /* n_points: MP/OMP dictionary columns, Np <= Ldict <= Nfft */
    const double* pilot_pattern_host;   /* 2 complex doubles: pilot q (0-based) carries pattern[q % 2] in every symbol */
    const uint32_t* payload_host;       /* packed payload bits; point k transmits the first S * Nd_k * bps of them */
    int64_t payload_bits;
    int32_t profile;                    /* as ofdm_tdl_channel: 0 EPA, 1 EVA, 2 ETU */
    double fs_hz;
    double snr_db;
    int64_t mc_runs;                    /* 1 .. 1,000,003 */
    int64_t tile_runs;                  /* runs per work item; 0 = 4096 (per run about 4 Nfft + 3 N_carrier complex of temporaries) */
    int32_t rank, world;
    uint64_t seed;
    double near_eps;                    /* symbols whose two smallest squared distances differ by less are counted */
    double tie_eps;                     /* OMP near-tie threshold, as ofdm_omp_ex */
} ofdm_part2_params;
/* nmse_dev: n_points x 4 x mc_runs doubles, [k][e][r] with e = LS, MMSE, MP, OMP; only this call's share is written.
 * counts_dev: n_points x 4 x 3 int64 += {bit errors, bits, symbols within near_eps of a decision boundary}.
 * runs_dev: n_points x 2 int64 += {runs processed, OMP runs with a near-tie}.  The values do not depend on the rank count
 * or the tile size; the caller sums the arrays of all ranks (each NMSE cell is written by one rank). */
OFDM_API int ofdm_sweep_part2(ofdm_ctx*, const ofdm_link_params* base, const ofdm_part2_params*, double* nmse_dev,
                              int64_t* counts_dev, int64_t* runs_dev);
/* Task-4 synchroniser and channel-estimate accuracy study over SNR (`Task 4/Main_model_Task_4.m:95-110,277-374`,
 * `Task 4/README.md:111-121,189-193`): per stream TX -> Noise -> add_STO -> add_CFO -> multipath -> the M2 RX chain of
 * ofdm_rx_chain_t4_ex (its split form, for any tile size), reporting the estimates, the channel-estimate error and the MER.
 * Share rule, stream numbering g = snr_index * streams_per_point + j, tiles and the Philox keys of the payload, noise and
 * STO / CFO draws are those of ofdm_sweep_ber's Task-4 chain: with sto_mode 0 and all three desync flags on, the same seed
 * transmits the same streams.  FP32 contexts and Nfft = 1024 only (OFDM_ERR_UNSUPPORTED otherwise); word-aligned streams.
 * rec_dev: n_snr x 9 x streams_per_point doubles, [i][f][j]; only this call's share is written.  Fields f:
 *   0 TgPosition (1-based, 65 on detector failure; 0 when time_desync = 0, the offset the chain then applies)
 *   1 FreqOffset (0 when freq_desync = 0)
 *   2 IFO (-1: no bin above 0.77, the chain then removes none; 0 when freq_desync = 0)
 *   3 tau, 4 phase_shift of fine_sync (0 when time_desync = freq_desync = 0)
 *   5 mean over k = 1..N_carrier of |H_est(k) - H(k)|^2, H = fft(h, Nfft)(1:N_carrier) of the taps in double (H = 1 without
 *     multipath); NaN when mp_desync = 0, or where the estimate itself is NaN (a failed synchronisation)
 *   6 MER_func of the stream's equalised data carriers in dB (`MER_func.m:7-25`)
 *   7 the true STO (nsto), 8 the true CFO
 * counts_dev: n_snr x 4 int64 += {bit errors, bits, guard-interval detector failures, streams with IFO = -1}.  The values
 * do not depend on the rank count or the tile size; the caller sums the arrays of all ranks (each record cell is written by
 * one rank). */
typedef struct ofdm_sync_params {
    int32_t n_snr;
    const double* snr_db_host;   /* n_snr SNR points in dB */
    int64_t streams_per_point;
    int64_t tile_streams;        /* streams per work item; 0 = 8192 (two signal buffers of tile x stream bytes are allocated) */
    int32_t rank, world;
    uint64_t seed;
    const double* taps_host;     /* n_taps x 2 doubles (delay, amplitude), delays integers in [0, Nfft); n_taps = 0: no multipath */
    int32_t n_taps;
    int32_t sto_mode;            /* 0: drawn as ofdm_sweep_ber (sto_max, cfo_int_max); 1: sto_fixed / cfo_fixed for every stream */
    int32_t sto_max, cfo_int_max;
    int32_t sto_fixed;
    double cfo_fixed;
    int32_t time_desync, freq_desync, mp_desync;   /* receiver stages, as ofdm_rx_chain_t4_ex */
} ofdm_sync_params;
OFDM_API int ofdm_sweep_sync(ofdm_ctx*, const ofdm_link_params*, const ofdm_sync_params*, double* rec_dev, int64_t* counts_dev);
/* Task-2 PAPR study (`Task 2/Main_model_Task_2.m:72-82`, `Task 2/README.md:54,69-71`): calculatePAPR of every transmitted
 * stream and the distribution of calculate_window_PAPR over all its windows, for points k = 0..n_points-1 that differ in the
 * scrambler flag and the payload.  Work item g = k * streams_per_point + j; the call processes the share
 * ofdm_sweep_share(n_points * streams_per_point, rank, world) gives, in tiles of tile_streams streams that never straddle a
 * point.  Stream (k, j) is the TX chain's serial stream of L = S * (Nfft + Tg) samples for `lp` with scramble =
 * scramble_host[k] (lp->scramble is ignored); no channel is applied.  The payload depends on j only, not on k, so a plain
 * and a scrambled point with the same p_one (or the same pool) transmit the same payloads -- a paired comparison:
 *   - Bernoulli (pool_host NULL): bit i of stream j is 1 iff u_i < floor(p_one_host[k] * 2^32), u_i = word i mod 4 of
 *     Philox4x32-10 at counter (i / 4, j) in a key space of its own -- the bits ofdm_payload_bernoulli writes;
 *   - pool: bit i of stream j is pool bit (j * pool_stride + i) mod pool_bits (packed, the library's bit layout).
 * papr_dev: n_points x streams_per_point doubles, [k][j] = calculatePAPR of the whole serial stream, cyclic prefixes included
 * (`calculatePAPR.m:2-11`); only this call's share is written.
 * hist_dev: n_points x n_bins int64, ADDED to (+=): every window of calculate_window_PAPR(x, Nfft) (length Nfft, step 1, L - Nfft
 * + 1 per stream), with v its value rounded to the context's real type exactly as ofdm_window_papr returns it, counts in bin
 * min(floor((double)v / bin_db), n_bins - 1); negative v (rounding) and NaN (an all-zero window) count in bin 0.  The CCDF at
 * edge b * bin_db -- the fraction of windows with bin >= b -- is therefore exact; ofdm_ccdf gives the exact ecdf of stored values.
 * The values do not depend on the rank count or the tile size; the caller sums both arrays over ranks (each PAPR cell is
 * written by one rank, the histogram is integer).  FP32 and FP64 contexts, any power-of-two Nfft of the TX chain;
 * OFDM_ERR_UNSUPPORTED when the statistics kernel's shared memory (2 Nfft (8 + sizeof(real)) + 4 n_bins bytes) exceeds the
 * device's limit per block (FP64 at Nfft 8192). */
typedef struct ofdm_papr_params {
    int32_t n_points;
    const int32_t* scramble_host;   /* n_points: 0 plain, 1 Scrambler with per-frame reset from lp->reg0_host */
    const double* p_one_host;       /* n_points: P(bit = 1) of the Philox payload, 0 < p < 1; ignored when pool_host is set */
    const uint32_t* pool_host;      /* optional packed payload pool (library bit layout), e.g. file_reader('eagle.tiff') */
    int64_t pool_bits;              /* 1 .. 2^32 when pool_host is set */
    int64_t pool_stride;            /* >= 0: stream j reads pool bits (j * pool_stride + i) mod pool_bits, i = 0 .. stream_bits-1 */
    int64_t streams_per_point;
    int64_t tile_streams;           /* 0 = 8192 (one signal buffer of tile x L complex samples is allocated) */
    int32_t rank, world;
    uint64_t seed;
    double bin_db;                  /* histogram bin width in dB, > 0 */
    int32_t n_bins;                 /* 1 .. 16384; the last bin also takes everything above it */
} ofdm_papr_params;
OFDM_API int ofdm_sweep_papr(ofdm_ctx*, const ofdm_link_params*, const ofdm_papr_params*, double* papr_dev, int64_t* hist_dev);
/* Task-3 BER and MER study over constellations and SNR (`Task 3/Main_model_Task_3.m:192-268`, `Task 3/README.md:53-55`): per
 * stream TX -> Noise -> add_STO -> add_CFO -> multipath -> OFDM_demodulator -> get_payload -> demapping -> DeScrambler -> BER
 * and MER_func.  Task 3 has no synchroniser, estimator or equaliser: the STO, CFO and multipath reach the decisions
 * uncorrected.  Point k has its own constellation, SNR and fixed STO / CFO.  From `lp` the call reads Nfft, Tg, N_carrier,
 * S, SpF, the carriers, reg0 and scramble; lp->constellation is ignored.  Stream g = k * streams_per_point + j; the call
 * processes the share ofdm_sweep_share(n_points * streams_per_point, rank, world) gives, in tiles that never straddle a point.
 * Stream g carries the first S * Nd * bps_k bits of the Philox words ofdm_payload_bits draws for it, as one contiguous
 * bitstream: these are the scrambled frames s, the payload is p = DeScrambler(s) (p = s when lp->scramble = 0), and the
 * transmitter maps s without scrambling.  The channel is ofdm_channel_t4_p with the point's SNR, STO and CFO, so a call whose
 * points share one constellation transmits, with equal pilot values, the streams ofdm_sweep_sync transmits for the same SNR
 * list, seed and taps with sto_mode 1.  The receiver decides every symbol in the pass that transforms it: its bins and
 * decisions are those of ofdm_rx_chain_t4_ex(..., 0, 0, 0, ...) when that call runs its split chain (>= 512 streams of a
 * shape whose fused kernel fits; its other kernels round differently).  FP32 contexts and Nfft = 1024 only, data carriers
 * within N_carrier (OFDM_ERR_UNSUPPORTED otherwise); streams need not be word aligned.
 * mer_dev: n_points x 2 x streams_per_point doubles, [k][f][j]: f = 0 the sum of |ideal|^2, f = 1 the sum of |ideal - rx|^2
 * over the stream's data symbols, so MER_func of the stream is 10 log10(f0 / f1) dB; only this call's share is written, and
 * each cell is summed in an order that depends on the stream shape only.
 * counts_dev: n_points x 3 int64 += {bit errors after DeScrambler, bits, symbols within near_eps of a decision boundary}.
 * The values do not depend on the rank count or the tile size; the caller sums both arrays over ranks (each MER cell is
 * written by one rank). */
typedef struct ofdm_mer_params {
    int32_t n_points;
    const int32_t* constellation_host; /* n_points: OFDM_BPSK .. OFDM_16QAM */
    const double* snr_db_host;         /* n_points; +INFINITY = noise-free (Noise.m's noise power is then 0); not NaN */
    double pilot_scale;                /* > 0: every pilot of point k is pilot_scale * max|constellation_func(c_k)|, real
                                          (Task 3's scalar broadcast, `Main_model_Task_3.m:57-59`); 0: lp->pilot_vals_host */
    const int32_t* nsto_host;          /* n_points or NULL (= 0): fixed add_STO offset, >= 0, not corrected */
    const double* cfo_host;            /* n_points or NULL (= 0): fixed add_CFO offset, finite, not corrected */
    const double* taps_host;           /* n_taps x 2 doubles (delay, amplitude), delays integers in [0, Nfft); n_taps = 0: no multipath */
    int32_t n_taps;
    int64_t streams_per_point;
    int64_t tile_streams;              /* streams per work item; 0 = 8192 (two signal buffers of tile x stream bytes are allocated) */
    int32_t rank, world;
    uint64_t seed;
    double near_eps;                   /* symbols whose two smallest squared distances differ by less are counted; 0 = off */
} ofdm_mer_params;
OFDM_API int ofdm_sweep_mer(ofdm_ctx*, const ofdm_link_params*, const ofdm_mer_params*, double* mer_dev, int64_t* counts_dev);
/* first / count of the contiguous share of `total_streams` that (rank, world) processes */
OFDM_API int ofdm_sweep_share(int64_t total_streams, int rank, int world, int64_t* first, int64_t* count);
/* The sweep's synthetic inputs, also usable on their own: payload words of streams first_stream_id .. +n_streams-1
 * (n_streams x words_per_stream uint32), and per-stream STO / CFO draws (either output may be NULL). */
OFDM_API int ofdm_payload_bits(ofdm_ctx*, uint32_t* bits_dev, int64_t n_streams, int64_t words_per_stream, uint64_t seed,
                               int64_t first_stream_id);
OFDM_API int ofdm_draw_sto_cfo(ofdm_ctx*, int64_t B, uint64_t seed, int64_t first_stream_id, int sto_max, int cfo_int_max,
                               int32_t* nsto_dev, double* cfo_dev);
/* The Bernoulli payload of ofdm_sweep_papr: streams first_stream_id .. +n_streams-1 of stream_bits bits each (any length,
 * not padded to words) as ONE contiguous bitstream, the input ofdm_tx_chain takes; OFDM_BIT_WORDS(n_streams * stream_bits)
 * words are written and the bits past the last stream are 0.  Bit i of stream j is 1 iff u_i < floor(p_one * 2^32), u_i =
 * word i mod 4 of Philox4x32-10 at counter (i / 4, j) in a key space of its own; 0 < p_one < 1. */
OFDM_API int ofdm_payload_bernoulli(ofdm_ctx*, uint32_t* bits_dev, int64_t n_streams, int64_t stream_bits, double p_one,
                                    uint64_t seed, int64_t first_stream_id);

/* ---- device groups: one call runs a sweep on several GPUs of the process ------------------------------------------------- */
/* A group holds one context per entry of `devices`, in the given order: member i is rank i of world n_devices.  Ids are CUDA
 * device ordinals (0-based) and may repeat -- two members on one GPU are two contexts there, valid and bit-identical.
 * ofdm_group_create returns OFDM_ERR_INVALID for n_devices <= 0, a NULL list or a bad precision, and OFDM_ERR_NODEVICE for an id
 * without an sm_100 device; on failure *out is NULL and nothing is left allocated.  The members are created on threads of their
 * own, so the calling thread's current device is what it was before.
 *
 * ofdm_group_sweep_* run the ofdm_sweep_* call of the same name on every member at once, one host thread per member for the
 * duration of the call.  The rank / world fields of the params are ignored (the group sets them); every other field means what
 * it means for the single-context call, and the same checks apply.  Outputs are HOST arrays of the shape and layout of the
 * single-context call's device arrays, and are overwritten (not added to):
 *   - integer arrays (counters, the PAPR histogram, part-2 runs) are the sum over the members;
 *   - per-stream / per-run cells (mse, rec, papr, nmse) are copied from the member whose ofdm_sweep_share range holds them, so
 *     -0.0 and NaN payloads survive;
 * the result is bit-identical to the single-context call with world = 1.  Each member zeroes its own device outputs, runs the
 * sweep on its own stream, copies its results back and synchronises; its device buffers are kept for the next call
 * (grow-only) and freed by ofdm_group_destroy.  Nothing is left running or enqueued when a call returns.  A member whose share
 * is empty (more members than streams) launches nothing and contributes zeros.
 * If a member fails, the call returns the status of the lowest-index failing member and ofdm_group_last_error reads
 * "device <id> (member <i>): <that member's ofdm_last_error>"; the host outputs are then unspecified and the group stays
 * usable.  One call at a time per group. */
typedef struct ofdm_group ofdm_group;
OFDM_API int ofdm_group_create(ofdm_group** out, const int* devices, int n_devices, int precision);
OFDM_API void ofdm_group_destroy(ofdm_group* g);   /* NULL: no-op */
OFDM_API const char* ofdm_group_last_error(const ofdm_group* g);
OFDM_API int ofdm_group_size(const ofdm_group* g);
/* counts_host: n_snr x 4 int64 */
OFDM_API int ofdm_group_sweep_ber(ofdm_group*, const ofdm_link_params*, const ofdm_sweep_params*, int64_t* counts_host);
/* mse_host: n_snr x 4 x streams_per_point doubles; counts_host: n_snr x 2 int64 */
OFDM_API int ofdm_group_sweep_mse(ofdm_group*, const ofdm_link_params*, const ofdm_sweep_params*, int Ldict, double* mse_host,
                                  int64_t* counts_host);
/* rec_host: n_snr x 9 x streams_per_point doubles; counts_host: n_snr x 4 int64 */
OFDM_API int ofdm_group_sweep_sync(ofdm_group*, const ofdm_link_params*, const ofdm_sync_params*, double* rec_host, int64_t* counts_host);
/* papr_host: n_points x streams_per_point doubles; hist_host: n_points x n_bins int64 */
OFDM_API int ofdm_group_sweep_papr(ofdm_group*, const ofdm_link_params*, const ofdm_papr_params*, double* papr_host, int64_t* hist_host);
/* mer_host: n_points x 2 x streams_per_point doubles; counts_host: n_points x 3 int64 */
OFDM_API int ofdm_group_sweep_mer(ofdm_group*, const ofdm_link_params*, const ofdm_mer_params*, double* mer_host, int64_t* counts_host);
/* nmse_host: n_points x 4 x mc_runs doubles; counts_host: n_points x 4 x 3 int64; runs_host: n_points x 2 int64 */
OFDM_API int ofdm_group_sweep_part2(ofdm_group*, const ofdm_link_params* base, const ofdm_part2_params*, double* nmse_host,
                                    int64_t* counts_host, int64_t* runs_host);

#ifdef __cplusplus
}
#endif
#endif /* OFDM_B200_H */
