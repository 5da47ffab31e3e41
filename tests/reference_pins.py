"""Numbers the REFERENCE ITSELF holds for the link chain (its READMEs and figures; it ships no tests), and the
experiment definitions that reproduce them.  Shared by `test_reference_pins.py` (oracle, CPU) and
`test_gpu_reference_pins.py` (CUDA path through the C ABI).  Citations are path:line under /root/reference.

What is pinned and how firmly
-----------------------------
P1  `Task 3/README.md:57-60`, figure `Task 3/graphs/ber(snr).png` (produced by `Task 3/Main_model_Task_3.m:192-268`,
    parameters as committed: Nfft 1024, 400 carriers, 15 % pilots all +4/3*max, 50 symbols, eagle.tiff payload,
    per-frame scrambler, AWGN only).  21 points read off the figure's log axis (reading error about +-5 %, plus the
    Monte-Carlo error of the reference's single 16,600*bps-bit run, see `ber_tolerance`).  Pins: constellation tables and bit labelling,
    scrambler/descrambler (the 3x error multiplication), `Noise.m`'s SNR convention, IFFT/FFT scaling, carrier layout.
P2  `Task 3/README.md:53-55`, figure `Task 3/graphs/info.png`: "SNR=25 dB; MER=29.0341 dB; BER=0".  The committed
    script (15 % pilots) gives 27.8 dB in the oracle; MER = SNR + 10 log10(Nfft / (Nd + Np a^2)) explains both: the
    README line was printed by a run with (almost) no pilots -- Np = 2 (`Percent_pilot` <= 0.25) gives 29.035 dB
    analytically.  Pins `Noise.m` + `MER_func.m` + FFT scaling under that INFERRED configuration (stated as such).
P3  `Task 4/README.md:179-183`: equalised MER 60 / 108 / 130 dB for linear / cubic / spline interpolation, noise-free,
    3-tap multipath `[0 1; 4 .6; 10 .3]` (`Task 4/Main_model_Task_4.m:252-256`).  With the committed 15 % pilots the
    oracle gives 42.7 / - / 94.2 dB; with pilot step 2 (`Percent_pilot = 50`; the README's own figure 23 is "pilot
    period = 2") it gives 59.8 / 106.9 / 130.1 dB on the carriers inside the uniform pilot run (carrier 399, which sits
    in the irregular last gap 397 -> 400, excluded; including it the spline figure drops to 123.2).  'cubic' is MATLAB's
    cubic convolution (Keys a = -1/2), which needs uniform pilots.  INFERRED configuration, stated as such.  Pins the
    channel model, LS estimate, not-a-knot spline, equaliser and `MER_func`.
P4  `Task 2/README.md:54`, figure `Task 2/graphs/PAPR1.png`: PAPR 23 dB unscrambled, 10 dB scrambled (printed with
    `int2str`; `Task 2/Main_model_Task_2.m:73-74`).  Oracle: 22.5 / 11.2 dB -- a peak statistic of one payload, so the
    pin is +-1.5 dB.
"""
import os
import struct

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

# P1: BER(SNR) read off Task 3/graphs/ber(snr).png
BER_SNR_FIGURE = {
    "BPSK": {0: 0.043, 2: 0.0095, 4: 0.00135},
    "QPSK": {0: 0.17, 2: 0.08, 4: 0.023, 6: 0.0036},
    "8PSK": {0: 0.34, 2: 0.26, 4: 0.175, 6: 0.093, 8: 0.038, 10: 0.010},
    "16QAM": {0: 0.42, 2: 0.37, 4: 0.30, 6: 0.215, 8: 0.125, 10: 0.054, 12: 0.016, 14: 0.0022},
}


BPS = {"BPSK": 1, "QPSK": 2, "8PSK": 3, "16QAM": 4}


def ber_tolerance(ber_fig, cname):
    """Relative tolerance on a figure reading: 5 % reading error + 2.5 sigma of the REFERENCE's own single run, which holds
    16,600*bps bits per point; descrambler errors come in triples, so it has about ber*bits/3 independent error events
    (BPSK at 0 dB: 238 events, sigma 6.5 %; 16QAM at 8 dB: 2,767 events, sigma 1.9 %)."""
    events = max(ber_fig * 16600 * BPS[cname] / 3.0, 1.0)
    return 0.05 + 2.5 / events ** 0.5


MER_AWGN_25DB = 29.0341            # P2
MER_TABLE_T4 = {"linear": 60.0, "cubic": 108.0, "spline": 130.0}     # P3
TAPS_T4 = [[0, 1], [4, .6], [10, .3]]
PAPR_T2 = {"plain": 23.0, "scrambled": 10.0}                         # P4


def eagle_bits(n):
    """First n payload bits of `file_reader('eagle.tiff', n)` from the committed golden input vector."""
    raw = np.frombuffer(open(os.path.join(HERE, "golden", "eagle_bits.bin"), "rb").read(), dtype=np.uint8)
    return np.unpackbits(raw)[:n].copy()


def write_eagle_tiff(path, side=360):
    """Write an 8-bit grey-level baseline TIFF (side x side, one uncompressed strip) whose Otsu binarisation, read
    column-major, is the golden payload.  The reference image is not part of this repository: each pixel's grey level is
    drawn (seeded) from a dark band for a 0 and a bright band for a 1, so every threshold in the gap between the bands
    gives back `eagle_bits(side * side)`."""
    bits = eagle_bits(side * side)
    rng = np.random.default_rng(360)
    grey = np.where(bits == 1, rng.integers(150, 256, bits.size), rng.integers(0, 100, bits.size)).astype(np.uint8)
    data = grey.reshape((side, side), order="F").tobytes()
    entries = [(256, 4, 1, side), (257, 4, 1, side), (258, 3, 1, 8), (259, 3, 1, 1), (262, 3, 1, 1), (273, 4, 1, 8),
               (277, 3, 1, 1), (278, 4, 1, side), (279, 4, 1, len(data))]
    ifd = struct.pack("<H", len(entries)) + b"".join(struct.pack("<HHII", *e) for e in entries) + struct.pack("<I", 0)
    with open(path, "wb") as fh:
        fh.write(b"II*\0" + struct.pack("<I", 8 + len(data)) + data + ifd)
    return str(path)


def keys_cubic(x, y, xq):
    """MATLAB interp1 'cubic' (= 'v5cubic', cubic convolution, uniform x) with its end extension 3y1-3y2+y3."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y)
    h = x[1] - x[0]
    ye = np.concatenate([[3 * y[0] - 3 * y[1] + y[2]], y, [3 * y[-1] - 3 * y[-2] + y[-3]]])
    s = (np.asarray(xq, dtype=np.float64) - x[0]) / h
    k = np.clip(np.floor(s).astype(int), 0, len(x) - 2)
    t = s - k
    return ((-t**3 + 2 * t**2 - t) * ye[k] + (3 * t**3 - 5 * t**2 + 2) * ye[k + 1] + (-3 * t**3 + 4 * t**2 + t) * ye[k + 2]
            + (t**3 - t**2) * ye[k + 3]) / 2
