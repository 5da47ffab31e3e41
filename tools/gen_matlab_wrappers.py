#!/usr/bin/env python
"""Generate matlab/<RefName>.m: wrappers with the reference's exact signatures (cited) that forward to
the MEX gateway.  Run from the repo root; the output is committed."""
import os

W = [
    ("Scrambler", "[sc_sequence, Register]", "Register, sequence", "Task 5/Scrambler.m:1"),
    ("DeScrambler", "[dsc_sequence, Register]", "Register, sequence", "Task 5/DeScrambler.m:1"),
    ("constellation_func", "[Dictionary, Bit_depth_Dict]", "Constellation", "Task 5/constellation_func.m:4"),
    ("mapping", "[IQ,pad]", "bits, constellation", "Task 5/mapping.m:1"),
    ("demapping", "[de_bits]", "pad, IQ, Constellation", "Task 5/demapping.m:1"),
    ("OFDM_map_carriers", "mapped_carriers", "QAM_payload, N_symb, Nfft, dataCarriers, pilotCarriers, pilotValues", "Task 5/OFDM_map_carriers.m:2"),
    ("OFDM_modulator", "OFDM_time_guarded", "OFDM_symbols, T_guard", "Task 5/OFDM_modulator.m:2"),
    ("OFDM_demodulator", "TX_IQ", "OFDM_time_guarded, T_guard", "Task 5/OFDM_demodulator.m:2"),
    ("get_payload", "RX_IQ", "RX_OFDM_symbols, dataCarriers", "Task 5/get_payload.m:2"),
    ("add_STO", "y_STO", "y, nSTO", "Task 5/add_STO.m:1"),
    ("add_CFO", "y_CFO", "y, CFO, Nfft", "Task 5/add_CFO.m:1"),
    ("Noise", "[IQ_RX, N_var]", "SNR, IQ_TX, varargin", "Task 5/Noise.m:1"),
    ("get_MP_channel_resp", "[impulse_response,frequency_response]", "channel_taps, Nfft", "Task 5/get_MP_channel_resp.m:2"),
    ("AutoCorrFunction", "[AutoCorr, TgPosition, FreqOffset]", "RxSignal, WidthWindow, Nfft", "Task 5/AutoCorrFunction.m:1"),
    ("remove_IFO", "[fixed_rx_signal, IFO]", "rx_signal, Nfft", "Task 5/remove_IFO.m:1"),
    ("fine_sync", "sync_signal", "rx_signal, pilotCarriers, pilotValues, time_desync, freq_desync", "Task 4/fine_sync.m:1"),
    ("estimate_channel", "[H_est,Hest_at_pilots]", "rx_signal, allCarriers, pilotCarriers, pilotValues", "Task 5/estimate_channel.m:1"),
    ("LS_CE", "[H_LS]", "Y, Xp, pilot_loc, N_carrier", "Task 5/LS_CE.m:1"),
    ("MMSE_CE", "[H_MMSE]", "Y, Xp, pilot_loc, Nfft, N_carrier, h, SNR", "Task 5/MMSE_CE.m:1"),
    ("interpolate", "[H_interpolated]", "H, pilot_loc, Nfft, method", "Task 5/interpolate.m:1"),
    ("equalize_signal", "equalized_Hest", "OFDM_demod, Hest, N_carrier", "Task 5/equalize_signal.m:1"),
    ("OMP_estimate", "[H_OMP,h_impulse_est,index]", "Y, sensing_matrix, Nfft, dominant_taps, SNR_dB", "Task 5/OMP_estimate.m:2"),
    ("MP_estimate", "[H_MP,h_impulse_est]", "Y, sensing_matrix, Nfft, dominant_taps", "Task 5/MP_estimate.m:2"),
    ("BER_func", "[BER]", "Bit_Tx, Bit_Rx", "Task 5/BER_func.m:1"),
    ("MER_func", "[MER]", "IQ_RX, Constellation", "Task 5/MER_func.m:1"),
    ("calculatePAPR", "PAPR", "OFDM_signal", "Task 5/calculatePAPR.m:2"),
    ("calculate_window_PAPR", "PAPRs", "Tx_OFDM_Signal, Nfft", "Task 5/calculate_window_PAPR.m:2"),
    ("calculateCCDF", "[PAPR_ccdf, CCDF]", "PAPR_values", "Task 5/calculateCCDF.m:2"),
]
NOTES = {
    "Noise": "%   Optional third argument: an L-by-2 matrix of unit normals (column 1 real part, column 2 imaginary\n"
             "%   part, the order of the reference's two normrnd calls) to share a realisation, or a scalar Philox seed.\n",
    "mapping": "%   bits is a column of 0/1 doubles; IQ is 1-by-N, pad = -1 when nothing was padded.\n",
    "OFDM_map_carriers": "%   pilotValues: Np-by-N_symb matrix, or a scalar (broadcast, as `Task 3/Main_model_Task_3.m:59` does).\n",
}
os.makedirs("matlab", exist_ok=True)
for name, outs, ins, cite in W:
    call_ins = ins.replace("varargin", "varargin{:}")
    if name in ("mapping", "demapping", "MER_func", "constellation_func"):
        # MATLAB string scalars ("16QAM") -> char for the gateway
        var = {"mapping": "constellation", "demapping": "Constellation", "MER_func": "Constellation", "constellation_func": "Constellation"}[name]
        call_ins = call_ins.replace(var, f"char({var})")
    if name == "interpolate":
        call_ins = call_ins.replace("method", "char(method)")
    n_out = outs.count(",") + 1
    lhs = outs if outs.startswith("[") else f"[{outs}]" if n_out > 1 else outs
    body = (f"function {outs} = {name}({ins})\n"
            f"%{name.upper()}  GPU (libofdm_b200, sm_100a) drop-in for `{cite}` of ladnlav/OFDM-course.\n"
            f"%   Same signature, shapes and orientation as the reference; forwards to the MEX gateway.\n"
            f"{NOTES.get(name, '')}"
            f"    {lhs} = ofdm_mex('{name}', {call_ins});\n"
            f"end\n")
    open(os.path.join("matlab", name + ".m"), "w").write(body)
open("matlab/OFDM_map_carriers_v1.m", "w").write(
    "function mapped_carriers = OFDM_map_carriers_v1(QAM_payload, N_symb, Nfft, dataCarriers, pilotCarriers, amp_pilots)\n"
    "%OFDM_MAP_CARRIERS_V1  Task-1/2 variant (`Task 1/OFDM_map_carriers.m:2`): alternating +a / a*exp(1i*pi) pilots,\n"
    "%   repmat(...,1,50).  Rename to OFDM_map_carriers.m when running the Task 1-2 scripts.\n"
    "    pv = zeros(1, length(pilotCarriers)); pv(1:2:end) = amp_pilots*exp(1i*0); pv(2:2:end) = amp_pilots*exp(1i*pi);\n"
    "    mapped_carriers = ofdm_mex('OFDM_map_carriers', QAM_payload, N_symb, Nfft, dataCarriers, pilotCarriers, repmat(pv', 1, 50));\n"
    "end\n")
open("matlab/apply_channel.m", "w").write(
    "function y = apply_channel(x, h)\n"
    "%APPLY_CHANNEL  conv(x, h.', 'full') truncated to length(x) (`Task 5/Main_model_Task_5.m:126-127`).\n"
    "    y = ofdm_mex('apply_channel', x, h);\n"
    "end\n")
# ---- batched / fused entries (no reference function of that name: they replace the script LOOPS)
BATCH = {
"ofdm_link.m": """function L = ofdm_link(P)
%OFDM_LINK  Pack the link description of a reference script into the positional list the batched MEX ops take.
%   P has the script's own variable names (`Task 5/Main_model_Task_5.m:6-46`): Nfft, T_Guard, N_carrier, N_symb,
%   Amount_ODFM_SpF, Constellation, dataCarriers, pilotCarriers, pilotValues (Np x N_symb or Np x 1), Register.
    L = {P.Nfft, P.T_Guard, P.N_carrier, P.N_symb, P.Amount_ODFM_SpF, char(P.Constellation), ...
         P.dataCarriers, P.pilotCarriers, P.pilotValues, P.Register};
end
""",
"ofdm_tx_chain.m": """function Tx = ofdm_tx_chain(P, bits)
%OFDM_TX_CHAIN  Scrambler (per-frame reset) -> mapping -> OFDM_map_carriers -> OFDM_modulator for B streams at once
%   (`Task 5/Main_model_Task_5.m:53-85` in one fused kernel).  bits: stream_bits x B of 0/1; Tx: (N_symb*(Nfft+T_Guard)) x B,
%   column b = the serial stream Tx_OFDM_Signal of stream b.
    L = ofdm_link(P);
    Tx = ofdm_mex('tx_chain', L{:}, bits);
end
""",
"ofdm_channel_t5.m": """function Rx = ofdm_channel_t5(Tx, SNR_dB, h, seed)
%OFDM_CHANNEL_T5  Noise then multipath for B streams (`Task 5/Main_model_Task_5.m:108,123-127`, one fused kernel).
%   Tx: L x B; SNR_dB: scalar, 1 x B or [] (no noise); h: impulse response from get_MP_channel_resp or [] (no multipath);
%   seed: Philox seed of the noise (stream b uses the counter stream (seed, b-1)).
    if nargin < 4, seed = 0; end
    Rx = ofdm_mex('channel_t5', Tx, SNR_dB, h, seed);
end
""",
"ofdm_channel_t4.m": """function Rx = ofdm_channel_t4(Tx, SNR_dB, nSTO, CFO, Nfft, h, seed)
%OFDM_CHANNEL_T4  Noise -> add_STO -> add_CFO -> multipath for B streams in one pass
%   (`Task 4/Main_model_Task_4.m:95,103,110,263-264`; the same samples as Noise, add_STO, add_CFO and conv called in turn).
%   Tx: L x B; SNR_dB, nSTO, CFO: scalars or 1 x B; h: impulse response from get_MP_channel_resp (1 for no multipath);
%   seed: Philox seed of the noise (stream b uses the counter stream (seed, b-1)).
    if nargin < 7, seed = 0; end
    Rx = ofdm_mex('channel_t4', Tx, SNR_dB, nSTO, CFO, Nfft, h, seed);
end
""",
"ofdm_rx_chain_t5.m": """function [bits, H, counts] = ofdm_rx_chain_t5(P, Rx, tx_bits, near_eps)
%OFDM_RX_CHAIN_T5  OFDM_demodulator -> LS_CE -> equalize_signal -> get_payload -> demapping -> DeScrambler -> BER count
%   for B streams in one pass (`Task 5/Task5_part2.m:169-174,269-303`).  Rx: L x B host matrix (the library chunks and
%   overlaps the transfers).  bits: stream_bits x B decided bits; H: N_carrier x B channel estimates;
%   counts = [bit errors, bits, symbols within near_eps of a decision boundary] (errors need tx_bits, else pass []).
    if nargin < 3, tx_bits = []; end
    if nargin < 4, near_eps = 0; end
    L = ofdm_link(P);
    [bits, H, counts] = ofdm_mex('rx_chain_t5', L{:}, Rx, tx_bits, near_eps);
end
""",
"ofdm_sweep_ber.m": """function counts = ofdm_sweep_ber(P, SNRs, streams_per_point, channel_taps, chain, seed, near_eps)
%OFDM_SWEEP_BER  The whole BER-vs-SNR Monte-Carlo loop on the GPU (`Task 3/Main_model_Task_3.m:192-268`,
%   `Task 5/Main_model_Task_5.m:303-346`; chain 'task4' adds the STO / CFO draws and the synchroniser of
%   `Task 4/Main_model_Task_4.m:95-110,277-366`).  counts: numel(SNRs) x 4 =
%   [bit errors, bits, near-boundary symbols, guard-interval detector failures]; BER = counts(:,1)./counts(:,2).
    if nargin < 5, chain = 'task5'; end
    if nargin < 6, seed = 1; end
    if nargin < 7, near_eps = 0; end
    L = ofdm_link(P);
    counts = ofdm_mex('sweep_ber', L{:}, SNRs, streams_per_point, channel_taps, char(chain), seed, near_eps);
end
""",
"ofdm_sweep_mse.m": """function [MSE, per_stream, counts] = ofdm_sweep_mse(P, SNRs, streams_per_point, channel_taps, seed, tie_eps, Ldict)
%OFDM_SWEEP_MSE  The channel-estimation MSE-vs-SNR loop of `Task 5/Main_model_Task_5.m:303-346` on the GPU: per stream
%   Noise -> multipath -> OFDM_demodulator -> LS_CE / MMSE_CE / MP_estimate / OMP_estimate and the MSE of each estimate
%   against the true response (`:195-205`).  P.dataCarriers = [] is the pilot-only comb-1 layout (`:24-33`).
%   MSE: numel(SNRs) x 4 means over the streams, columns LS, MMSE, MP, OMP; per_stream: streams_per_point x 4 x numel(SNRs);
%   counts: numel(SNRs) x 2 = [streams, OMP frames with a near-tie below tie_eps].  Ldict defaults to ceil(N_carrier/comb).
    if nargin < 5, seed = 1; end
    if nargin < 6, tie_eps = 0; end
    L = ofdm_link(P);
    if nargin < 7
        [MSE, per_stream, counts] = ofdm_mex('sweep_mse', L{:}, SNRs, streams_per_point, channel_taps, seed, tie_eps);
    else
        [MSE, per_stream, counts] = ofdm_mex('sweep_mse', L{:}, SNRs, streams_per_point, channel_taps, seed, tie_eps, Ldict);
    end
    per_stream = reshape(per_stream, streams_per_point, 4, numel(SNRs));
end
""",
"ofdm_sweep_part2.m": """function [NMSE, BER, per_run, counts, runs] = ofdm_sweep_part2(P, pilots, amp_pilots, bits, profile, fs, SNR, ...
                                                              monteCarloRuns, seed, near_eps, tie_eps, Ldict)
%OFDM_SWEEP_PART2  The pilot-density study of `Task 5/Task5_part2.m:46-321` on the GPU in one call: for every pilot layout and
%   monteCarloRuns static fading runs (lteFadingChannel stand-in, profile 'EPA' / 'EVA' / 'ETU' at sampling rate fs), the NMSE
%   of the LS / MMSE / MP / OMP estimates and the BER after equalising with each (`:148-304`).  P: Nfft, T_Guard, N_carrier,
%   N_symb, Amount_ODFM_SpF, Constellation.  pilots: a vector of combs (pilots 1:comb:N_carrier, `:50-55`) or a cell array of
%   pilot vectors (random masks, `:57-65`).  bits: 0/1 payload, at least the longest stream of any layout.
%   NMSE, BER: 4 x numel(pilots), rows LS, MMSE, MP, OMP (`:305-314`); per_run: monteCarloRuns x 4 x numel(pilots);
%   counts: 3 x 4 x numel(pilots) = [bit errors; bits; symbols within near_eps of a decision boundary];
%   runs: 2 x numel(pilots) = [runs; OMP runs with a near-tie below tie_eps].  Ldict defaults to ceil(Nfft/comb) for combs
%   and Nfft for pilot vectors.
    if nargin < 9, seed = 1; end
    if nargin < 10, near_eps = 0; end
    if nargin < 11, tie_eps = 0; end
    if nargin < 12, Ldict = []; end
    pv = [amp_pilots*exp(1i*0), amp_pilots*exp(1i*pi)]';                % `Task5_part2.m:86-91`: pilot q carries pv(mod(q-1,2)+1)
    if iscell(pilots)
        offsets = [0, cumsum(cellfun(@numel, pilots(:)'))];
        carriers = cell2mat(cellfun(@(v) v(:)', pilots(:)', 'UniformOutput', false));
    else
        carriers = pilots; offsets = [];
    end
    [NMSE, BER, per_run, counts, runs] = ofdm_mex('sweep_part2', P.Nfft, P.T_Guard, P.N_carrier, P.N_symb, P.Amount_ODFM_SpF, ...
        char(P.Constellation), carriers, offsets, Ldict, pv, bits, char(profile), fs, SNR, monteCarloRuns, seed, near_eps, tie_eps);
    n = size(NMSE, 2);
    per_run = reshape(per_run, monteCarloRuns, 4, n);
    counts = reshape(counts, 3, 4, n);
end
""",
"ofdm_sweep_sync.m": """function [rec, counts] = ofdm_sweep_sync(P, SNRs, streams_per_point, channel_taps, seed, sto, cfo, desync)
%OFDM_SWEEP_SYNC  Task 4's synchroniser and channel-estimate study over SNR on the GPU (`Task 4/Main_model_Task_4.m:95-110,
%   277-374`, `Task 4/README.md:111-121,189-193`): per stream Noise -> add_STO -> add_CFO -> multipath -> AutoCorrFunction ->
%   remove_IFO -> fine_sync -> estimate_channel -> equalize_signal -> demapping -> DeScrambler, reporting the estimates.
%   channel_taps: K x 2 (delay, amplitude) or [] for no multipath.  sto / cfo: the STO and CFO of every stream, or sto = []
%   to draw them as ofdm_sweep_ber does (cfo defaults to 0 with a given sto) (Time_Delay = randi([0, Nfft + T_Guard]), Freq_Shift = randi([0, 30]) + rand - 0.5).
%   desync: [time_desync freq_desync mp_desync] (default [1 1 1]).
%   rec: streams_per_point x 9 x numel(SNRs), fields TgPosition, FreqOffset, IFO, tau, phase_shift, mean |H_est - H|^2 over
%   the carriers (NaN without mp_desync or where the estimate is NaN), MER_func in dB, true STO, true CFO.
%   counts: numel(SNRs) x 4 = [bit errors, bits, detector failures (TgPosition = 65), streams with IFO = -1].
    if nargin < 5, seed = 1; end
    if nargin < 6 || isempty(sto), sto = -1; cfo = 0; end
    if nargin < 7, cfo = 0; end
    if nargin < 8, desync = [1 1 1]; end
    L = ofdm_link(P);
    [rec, counts] = ofdm_mex('sweep_sync', L{:}, SNRs, streams_per_point, channel_taps, seed, sto, cfo, desync);
    rec = reshape(rec, streams_per_point, 9, numel(SNRs));
end
""",
"ofdm_sweep_papr.m": """function [CCDF, edges, hist, PAPR] = ofdm_sweep_papr(P, scramble, p_one, streams_per_point, seed, bin_db, n_bins, pool_bits, pool_stride)
%OFDM_SWEEP_PAPR  Task 2's PAPR study on the GPU (`Task 2/Main_model_Task_2.m:72-82`): per point k the TX chain with
%   scramble(k) on streams_per_point payloads, calculatePAPR of every stream and the distribution of calculate_window_PAPR
%   over all windows.  p_one(k): P(bit = 1) of the Philox payload; or pool_bits: 0/1 payload bits (e.g. file_reader's), stream j
%   transmitting bits mod(j * pool_stride + (0 : stream_bits - 1), numel(pool_bits)) + 1 (p_one is then ignored).  Points with
%   the same payload source transmit the same payloads.
%   hist: n_bins x numel(scramble) window counts in bins of bin_db dB (the last bin takes everything above it);
%   edges = (0 : n_bins - 1)' * bin_db; CCDF(b, k) = fraction of point k's windows with PAPR >= edges(b), so
%   semilogy(edges, CCDF) draws what plot_custom_ccdf draws.  PAPR: streams_per_point x numel(scramble), calculatePAPR in dB.
    if nargin < 5, seed = 1; end
    if nargin < 6, bin_db = 0.01; end
    if nargin < 7, n_bins = 4000; end
    if nargin < 8, pool_bits = []; end
    if nargin < 9, pool_stride = 0; end
    L = ofdm_link(P);
    [hist, PAPR] = ofdm_mex('sweep_papr', L{:}, scramble, p_one, streams_per_point, seed, bin_db, n_bins, pool_bits, pool_stride);
    edges = (0 : n_bins - 1)' * bin_db;
    tail = flipud(cumsum(flipud(hist), 1));
    CCDF = tail ./ max(tail(1, :), 1);
end
""",
}
for fn, body in BATCH.items():
    open(os.path.join("matlab", fn), "w").write(body)
os.makedirs("matlab/examples", exist_ok=True)
open("matlab/examples/main_model_task5_batched.m", "w").write("""% Task-5 main loop, batched: what `Task 5/Main_model_Task_5.m:303-346` (BER over SNR for the LS estimator) does one
% stream and one SNR point at a time, here B streams per call and then the whole sweep in one call.
% Needs ofdm_mex on the path (see INTEGRATION.md) and an sm_100 GPU; not executable in the authoring image.
P.Nfft = 4096; P.N_carrier = 1024; P.T_Guard = P.Nfft / 8;
P.Amount_OFDM_Frames = 2; P.Amount_ODFM_SpF = 7; P.N_symb = P.Amount_OFDM_Frames * P.Amount_ODFM_SpF;
comb = 4;
P.pilotCarriers = 1:comb:P.N_carrier;                                   % `Main_model_Task_5.m:18-22`
P.dataCarriers = setdiff(1:P.N_carrier, P.pilotCarriers);
P.Constellation = "16QAM";
[dict, bps] = constellation_func(P.Constellation);
amp_pilots = 2 * max(abs(dict));                                        % `Task5_part2.m:86-91`
pv = zeros(1, numel(P.pilotCarriers)); pv(1:2:end) = amp_pilots * exp(1i * 0); pv(2:2:end) = amp_pilots * exp(1i * pi);
P.pilotValues = repmat(pv', 1, P.N_symb);
P.Register = [1 0 0 1 0 1 0 1 0 0 0 0 0 0 0];
channel_taps = [0 1; 4 .8; 10 .6; 15 .4; 21 .2; 25 .1];                 % `Main_model_Task_5.m:112-119`
[h, ~] = get_MP_channel_resp(channel_taps, P.Nfft);

% (1) explicit batch: B streams through TX -> channel -> RX, three calls
B = 64; stream_bits = P.N_symb * numel(P.dataCarriers) * bps;
bits = double(rand(stream_bits, B) > 0.5);
Tx = ofdm_tx_chain(P, bits);
Rx = ofdm_channel_t5(Tx, 20, h, 1);
[rx_bits, H, counts] = ofdm_rx_chain_t5(P, Rx, bits, 1e-4);
fprintf('B = %d streams at 20 dB: BER = %g (%d near-boundary symbols)\n', B, counts(1) / counts(2), counts(3));

% (2) the whole Monte-Carlo sweep in one call (payload, noise and channel generated on the GPU)
SNRs = 0:0.5:30;                                                        % `Task 3/Main_model_Task_3.m:192`
c = ofdm_sweep_ber(P, SNRs, 1024, channel_taps, 'task5', 1, 1e-4);
semilogy(SNRs, c(:, 1) ./ c(:, 2), 'LineWidth', 2); grid on; xlabel('SNR (dB)'); ylabel('BER');
""")
print(len(os.listdir("matlab")), "wrappers")
