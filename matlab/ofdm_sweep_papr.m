function [CCDF, edges, hist, PAPR] = ofdm_sweep_papr(P, scramble, p_one, streams_per_point, seed, bin_db, n_bins, pool_bits, pool_stride)
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
