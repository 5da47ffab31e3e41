function [MSE, per_stream, counts] = ofdm_sweep_mse(P, SNRs, streams_per_point, channel_taps, seed, tie_eps, Ldict)
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
