function [NMSE, BER, per_run, counts, runs] = ofdm_sweep_part2(P, pilots, amp_pilots, bits, profile, fs, SNR, ...
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
