function [BER, MER, per_stream, counts] = ofdm_sweep_mer(P, constellations, SNRs, streams_per_point, channel_taps, seed, sto, cfo, pilot_scale)
%OFDM_SWEEP_MER  Task 3's BER and MER study on the GPU (`Task 3/Main_model_Task_3.m:192-268`, `Task 3/README.md:53-55`): per
%   stream Noise -> add_STO -> add_CFO -> multipath -> OFDM_demodulator -> get_payload -> demapping -> DeScrambler -> BER_func,
%   and MER_func, with no synchroniser or equaliser (the STO, CFO and multipath are not corrected).  Point k is
%   (constellations{k}, SNRs(k)); constellations: a cell array of the reference's names ('BPSK', 'QPSK', '8PSK', '16QAM') or
%   one name for every point; SNR Inf is noise-free.  channel_taps: K x 2 (delay, amplitude) or [] for no multipath.
%   sto / cfo: the fixed STO and CFO, one value or one per point (default 0).  pilot_scale > 0: every pilot of point k is
%   pilot_scale * max(abs(constellation_func(constellations{k}))) (Task 3's scalar pilots, 4/3 there); 0 (default): P's pilots.
%   BER, MER: numel(SNRs) x 1; MER is MER_func over all streams of the point in dB.  per_stream: streams_per_point x 2 x
%   numel(SNRs), the sums of |ideal|^2 and |ideal - rx|^2 of each stream (its MER_func is 10*log10(f0 / f1)).
%   counts: numel(SNRs) x 3 = [bit errors, bits, symbols near a decision boundary].
    if nargin < 6, seed = 1; end
    if nargin < 7 || isempty(sto), sto = 0; end
    if nargin < 8 || isempty(cfo), cfo = 0; end
    if nargin < 9, pilot_scale = 0; end
    if ischar(constellations), constellations = repmat({constellations}, 1, numel(SNRs)); end
    ids = cellfun(@(c) find(strcmp(c, {'BPSK', 'QPSK', '8PSK', '16QAM'})), constellations);
    L = ofdm_link(P);
    [per_stream, counts] = ofdm_mex('sweep_mer', L{:}, double(ids), SNRs, streams_per_point, channel_taps, seed, sto, cfo, pilot_scale, 0);
    per_stream = reshape(per_stream, streams_per_point, 2, numel(SNRs));
    BER = counts(:, 1) ./ max(counts(:, 2), 1);
    MER = 10 * log10(squeeze(sum(per_stream(:, 1, :), 1)) ./ squeeze(sum(per_stream(:, 2, :), 1)));
    MER = MER(:);
end
