"""Pins P5 and P6 (DESIGN §2): the two Task-4 results of `Task 4/README.md` that the BER pins do not cover.  P6 is checked on
the float64 oracle here and with the same bounds on ofdm_sweep_sync in tests/test_gpu_sweep_sync.py; P5 is a GPU-vs-oracle
pin (tests/test_gpu_sweep_sync.py::test_p5_h_error_matches_oracle), and this file runs its experiment on the oracle.

P5, channel-estimate error over SNR at pilot step 4 (`Task 4/graphs/nmse(snr).png`, `README.md:189-193`): params_task4 at
25 % pilots (101 pilots, step 4, Nd 299), Noise then the 3-tap channel, no STO / CFO, the receiver without its sync stages;
error = mean over carriers 1..400 of |H_est - H|^2.  The figure reads about 5.5e-3 / 4e-4 / 1e-4 at 0 / 10 / 15 dB.  With 30
oracle streams per point the unnormalised error is 4.9e-3 / 4.8e-4 / 1.55e-4 (ratios 0.88 / 1.20 / 1.55 to the figure) and
the error divided by mean |H|^2 = 1.41 is 3.4e-3 / 3.4e-4 / 1.1e-4 (ratios 0.63 / 0.85 / 1.10): neither stays within a
factor of 1.5 at all three points.  So the figure is not pinned: its values are recorded below as documented numbers, and
P5 pins the GPU path's per-stream error against the oracle's on the same streams, at relative tolerance P5_RTOL.  Here the
oracle experiment is only checked to run on the layout the figure uses and to fall with SNR.

P6, CFO-estimator validity (`README.md:111-121`): params_task4, STO 150, CFO 0.24, no multipath, AutoCorrFunction.  On the
oracle (40 streams per point): at 0 dB every stream falls back to TgPosition = 65; from 5 dB on none does, and the largest
|FreqOffset - 0.24| is 0.014 at 5 and 10 dB, 0.009 at 15 dB and 0.004 at 20 dB.  The pin: at 0 dB at least 90 % of the
streams fall back; at 10 and 15 dB none does and |FreqOffset - 0.24| < 0.02 for at least 99 % of them.
"""
import numpy as np

import oracle as O
from oracle import chains as OC
from oracle import functions as F

TAPS4 = [[0, 1], [4, .6], [10, .3]]
P5_SNR = (0.0, 10.0, 15.0)
P5_FIGURE_MSE = (5.5e-3, 4e-4, 1e-4)     # read off the figure; documented, not asserted
# FP32 tolerance of the GPU-vs-oracle pin: the FP32 estimate carries rounding errors of about 1e-6 |H| (1,024-point FFT,
# pilot averaging, spline), against an estimation error |H_est - H| of about 1e-2 at 15 dB: about 2e-4 of the squared error
P5_RTOL = 1e-3
P6_FAIL_AT_0DB = 0.9
P6_CFO_BOUND = 0.02


def test_p5_channel_estimate_error_over_snr():
    p = OC.params_task4(percent=25)
    assert len(p.pilotCarriers) == 101 and len(p.dataCarriers) == 299 and p.pilotCarriers[1] - p.pilotCarriers[0] == 4
    h, _ = O.get_MP_channel_resp(TAPS4, p.Nfft)
    H = np.fft.fft(h, p.Nfft)[:p.N_carrier]
    rng = np.random.default_rng(50)
    means = []
    for snr in P5_SNR:
        err = []
        for _ in range(8):
            bits = rng.integers(0, 2, p.stream_bits).astype(np.uint8)
            tx, _, _ = OC.tx_chain(p, bits)
            rx = OC.impair_task4(p, tx, SNR_dB=snr, taps=TAPS4, rng=rng)
            r = OC.rx_chain_task4(p, rx, bits, time_desync=False, freq_desync=False)
            err.append(np.mean(np.abs(r["H"][:p.N_carrier] - H) ** 2))
        assert np.all(np.isfinite(err))
        means.append(np.mean(err))
    assert means[0] > means[1] > means[2], means


def test_p6_cfo_estimator_validity():
    p = OC.params_task4()
    rng = np.random.default_rng(60)
    for snr in (0.0, 10.0, 15.0):
        tg, fo = [], []
        for _ in range(10):
            bits = rng.integers(0, 2, p.stream_bits).astype(np.uint8)
            tx, _, _ = OC.tx_chain(p, bits)
            rx = OC.impair_task4(p, tx, SNR_dB=snr, Time_Delay=150, Freq_Shift=0.24, rng=rng)
            _, t, f = F.AutoCorrFunction(rx, p.T_Guard, p.Nfft)
            tg.append(t)
            fo.append(f)
        tg, fo = np.array(tg), np.array(fo)
        if snr == 0.0:
            assert np.mean(tg == 65) >= P6_FAIL_AT_0DB
        else:
            assert np.all(tg != 65)
            assert np.mean(np.abs(fo - 0.24) < P6_CFO_BOUND) >= 0.99
