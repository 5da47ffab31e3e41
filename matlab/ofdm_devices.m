function ids = ofdm_devices(ids)
%OFDM_DEVICES  The GPUs the six sweep wrappers run on: ofdm_sweep_ber, ofdm_sweep_mse, ofdm_sweep_sync, ofdm_sweep_mer,
%   ofdm_sweep_papr and ofdm_sweep_part2.  ids are 0-based CUDA device indices (as nvidia-smi lists them), not MATLAB's 1-based gpuDevice indices.
%   ofdm_devices(0:7) spreads every later sweep call over eight GPUs in this one MATLAB process, one share of the streams per
%   GPU; the results are bit-identical to the default ofdm_devices(0), one GPU.  An id may repeat.  ofdm_devices() returns
%   the current set.  Everything else (ofdm_tx_chain, ofdm_rx_chain_t5, the reference drop-ins) stays on device 0.
%   Bad ids raise ofdm:devices:*; ofdm_mex('precision', ...) keeps the set.
    if nargin < 1
        ids = ofdm_mex('devices');
    else
        ids = ofdm_mex('devices', double(ids));
    end
end
