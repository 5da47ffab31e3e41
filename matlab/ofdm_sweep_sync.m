function [rec, counts] = ofdm_sweep_sync(P, SNRs, streams_per_point, channel_taps, seed, sto, cfo, desync)
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
