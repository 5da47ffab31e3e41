"""Float64 restatement of the reference's link-chain functions (test infrastructure).

PARITY UNPINNED (see ``oracle/__init__.py``): no reference golden vectors exist and
MATLAB/Octave are absent, so this file is pinned on hand-derived KATs only.

Conventions kept from MATLAB so call sites read like the reference scripts:
  * carrier / pilot / tap index vectors are **1-based**;
  * matrices are ``(Nfft, N_symb)`` and are flattened column-major (``order='F'``);
  * vectors are returned 1-D (row/column orientation is noted in the docstring);
  * bits are arrays of 0/1 (any numeric dtype).
All citations are ``path:line`` under ``/root/reference/``.
"""
from __future__ import annotations

import numpy as np
from scipy.interpolate import CubicSpline

__all__ = [
    "Scrambler", "DeScrambler", "constellation_func", "mapping", "demapping",
    "OFDM_map_carriers", "OFDM_map_carriers_v1", "OFDM_modulator", "OFDM_demodulator",
    "get_payload", "add_STO", "add_CFO", "Noise", "get_MP_channel_resp", "apply_channel",
    "AutoCorrFunction", "remove_IFO", "fine_sync", "estimate_channel", "LS_CE", "MMSE_CE",
    "interpolate", "equalize_signal", "OMP_estimate", "MP_estimate", "BER_func", "MER_func",
    "interp1_spline", "sensing_matrix_dft", "pilot_layout_percent", "pilot_layout_comb",
    "calculatePAPR", "calculate_window_PAPR", "calculateCCDF", "DEFAULT_REGISTER",
    "Scrambler_fast", "DeScrambler_fast", "near_margin",
]

#: initial scrambler register used by every script (`Task 4/Main_model_Task_4.m:43`)
DEFAULT_REGISTER = np.array([1, 0, 0, 1, 0, 1, 0, 1, 0, 0, 0, 0, 0, 0, 0], dtype=np.uint8)


# --------------------------------------------------------------------------- a1/a2
def _array_xor(register):
    """`Task 5/Scrambler.m:18-28`: mask ``coeff_mask(2:end)`` (14 long) over the 15-cell
    register selects cells 13 and 14 (1-based)."""
    return int(register[12]) ^ int(register[13])


def Scrambler(Register, sequence):
    """`Task 5/Scrambler.m:1-16` -- multiplicative scrambler, feedback = scrambled bit.
    Returns ``(sc_sequence, Register)`` (final register, as the reference does)."""
    reg = [int(b) & 1 for b in np.asarray(Register).ravel()]
    seq = np.asarray(sequence).ravel()
    out = np.zeros(seq.size, dtype=np.uint8)
    for i in range(seq.size):
        symbol = (reg[12] ^ reg[13]) ^ (int(seq[i]) & 1)      # :8-9
        out[i] = symbol                                         # :11
        reg = [symbol] + reg[:-1]                               # :13-14 circshift + overwrite
    return out, np.array(reg, dtype=np.uint8)


def DeScrambler(Register, sequence):
    """`Task 5/DeScrambler.m:1-16` -- FIR inverse, feedback = received bit."""
    reg = [int(b) & 1 for b in np.asarray(Register).ravel()]
    seq = np.asarray(sequence).ravel()
    out = np.zeros(seq.size, dtype=np.uint8)
    for i in range(seq.size):
        feedback = int(seq[i]) & 1                              # :8
        out[i] = (reg[12] ^ reg[13]) ^ feedback                 # :9-10
        reg = [feedback] + reg[:-1]                             # :12-13
    return out, np.array(reg, dtype=np.uint8)


def DeScrambler_fast(Register, sequence):
    """Vectorised DeScrambler (same result as the loop above; used where the oracle is *timed* so the
    CPU baseline is not dominated by a Python per-bit loop): out[i] = in[i] ^ in[i-13] ^ in[i-14]
    with pre-history in[-m] = Register(m)."""
    reg = np.asarray(Register).ravel().astype(np.uint8) & 1
    seq = np.asarray(sequence).ravel().astype(np.uint8) & 1
    ext = np.concatenate([reg[::-1], seq])                      # ext[15 + i] = in[i], ext[15 - m] = Register(m)
    out = seq ^ ext[15 - 13: 15 - 13 + seq.size] ^ ext[15 - 14: 15 - 14 + seq.size]
    tail = np.concatenate([reg[::-1], seq])[::-1][:15]
    return out, tail.astype(np.uint8)


def Scrambler_fast(Register, sequence):
    """Vectorised Scrambler via the GF(2) identity 1/(1+p) = prod_j (1 + p^(2^j)), p = x^13 + x^14
    (SURVEY KAT 2); same result as the loop above."""
    reg = np.asarray(Register).ravel().astype(np.uint8) & 1
    t = (np.asarray(sequence).ravel().astype(np.uint8) & 1).copy()
    L = t.size
    for i in range(min(14, L)):                                  # fold the register pre-history into the input
        a = reg[12 - i] if 12 - i >= 0 else 0
        b = reg[13 - i] if 13 - i >= 0 else 0
        t[i] ^= a ^ b
    j = 0
    while (13 << j) < L:
        s13, s14 = 13 << j, 14 << j
        u = t.copy()
        u[s13:] ^= t[:L - s13]
        if s14 < L:
            u[s14:] ^= t[:L - s14]
        t = u
        j += 1
    tail = np.concatenate([reg[::-1], t])[::-1][:15]
    return t, tail.astype(np.uint8)


# --------------------------------------------------------------------------- a3
def constellation_func(Constellation):
    """`Task 5/constellation_func.m:4-29` -> (Dictionary (unit mean power), bits/symbol)."""
    name = str(Constellation)
    if name == "BPSK":
        d = np.array([-1 + 0j, 1 + 0j])
        bps = 1
    elif name == "QPSK":
        d = np.array([-1 - 1j, -1 + 1j, 1 - 1j, 1 + 1j])
        bps = 2
    elif name == "8PSK":
        gray_map = np.array([5, 4, 2, 3, 6, 7, 1, 0], dtype=np.float64)
        d = np.exp(1j * (gray_map * 2 * np.pi / 8))
        bps = 3
    elif name == "16QAM":
        d = np.array([-3 + 3j, -3 + 1j, -3 - 3j, -3 - 1j, -1 + 3j, -1 + 1j, -1 - 3j, -1 - 1j,
                      3 + 3j, 3 + 1j, 3 - 3j, 3 - 1j, 1 + 3j, 1 + 1j, 1 - 3j, 1 - 1j])
        bps = 4
    else:
        raise ValueError(f"unknown constellation {name!r}")
    norm = np.sqrt(np.sum(d * np.conj(d)) / d.size)           # :27-28
    return d / norm, bps


# --------------------------------------------------------------------------- a4/a5
def mapping(bits, constellation):
    """`Task 5/mapping.m:1-25` -> (IQ row vector, pad); pad = -1 when nothing was padded."""
    dictionary, bps = constellation_func(constellation)
    bits = np.asarray(bits).ravel().astype(np.int64)
    pad = -1
    rem = bits.size % bps
    if rem != 0:
        pad = bps - rem                                         # :10
        bits = np.concatenate([bits, np.zeros(pad, dtype=np.int64)])
    groups = bits.reshape(-1, bps)                              # :15
    weights = 1 << np.arange(bps - 1, -1, -1)                   # :18 'left-msb'
    idx = groups @ weights
    return dictionary[idx], pad


def demapping(pad, IQ, Constellation):
    """`Task 5/demapping.m:1-25` -- min squared-Euclid distance, first index on ties,
    MATLAB ``min`` skips NaN (all-NaN column -> index 1)."""
    dictionary, bps = constellation_func(Constellation)
    IQ = np.asarray(IQ).ravel()
    dist = (IQ.real[None, :] - dictionary.real[:, None]) ** 2 + \
           (IQ.imag[None, :] - dictionary.imag[:, None]) ** 2  # :9
    dist = np.where(np.isnan(dist), np.inf, dist)
    idx = np.argmin(dist, axis=0)                               # :12 (first min)
    shifts = np.arange(bps - 1, -1, -1)
    bits = ((idx[:, None] >> shifts[None, :]) & 1).astype(np.uint8).ravel()  # :15 int2bit MSB first
    if pad != -1:
        bits = bits[: bits.size - pad]                          # :21-23
    return bits


def near_margin(iq, Constellation):
    """Decision margin of each symbol of ``demapping``: second-smallest minus smallest squared
    distance to the constellation points, in float64 (0 on a decision boundary).  This is the
    quantity the device demappers compare with ``near_eps`` (not a reference function)."""
    dictionary, _ = constellation_func(Constellation)
    IQ = np.asarray(iq).ravel().astype(np.complex128)
    dist = (IQ.real[None, :] - dictionary.real[:, None]) ** 2 + (IQ.imag[None, :] - dictionary.imag[:, None]) ** 2
    two = np.partition(dist, 1, axis=0)[:2]
    return two[1] - two[0]


# --------------------------------------------------------------------------- a6
def OFDM_map_carriers(QAM_payload, N_symb, Nfft, dataCarriers, pilotCarriers, pilotValues):
    """`Task 5/OFDM_map_carriers.m:2-8` (v2). ``pilotValues`` is (Np, N_symb) or a scalar."""
    dataCarriers = np.asarray(dataCarriers, dtype=np.int64)
    pilotCarriers = np.asarray(pilotCarriers, dtype=np.int64)
    out = np.zeros((Nfft, N_symb), dtype=np.complex128)
    if dataCarriers.size:
        data = np.asarray(QAM_payload).ravel().reshape((dataCarriers.size, N_symb), order="F")
        out[dataCarriers - 1, :] = data                         # :6
    pv = np.asarray(pilotValues)
    out[pilotCarriers - 1, :] = pv if pv.ndim == 0 else pv.reshape(pilotCarriers.size, -1)  # :8
    return out


def OFDM_map_carriers_v1(QAM_payload, N_symb, Nfft, dataCarriers, pilotCarriers, amp_pilots):
    """`Task 1/OFDM_map_carriers.m:2-12` (v1): alternating +a / -a pilots built inside
    (``a*exp(1i*pi)`` keeps its ~1.2e-16 imaginary part); ``repmat(.,1,50)`` hard-codes 50
    columns, so N_symb must be 50 exactly as in the reference."""
    pilotCarriers = np.asarray(pilotCarriers, dtype=np.int64)
    pv = np.zeros(pilotCarriers.size, dtype=np.complex128)
    pv[0::2] = amp_pilots * np.exp(1j * 0)
    pv[1::2] = amp_pilots * np.exp(1j * np.pi)
    pv = np.tile(np.conj(pv)[:, None], (1, 50))                 # :11  pilotValues' is the ctranspose
    if N_symb != 50:
        raise ValueError("Task-1 OFDM_map_carriers hard-codes 50 symbols")
    return OFDM_map_carriers(QAM_payload, N_symb, Nfft, dataCarriers, pilotCarriers, pv)


# --------------------------------------------------------------------------- a7-a9
def OFDM_modulator(OFDM_symbols, T_guard):
    """`Task 5/OFDM_modulator.m:2-10`: column IFFT (1/N) + prepend last T_guard rows."""
    t = np.fft.ifft(np.asarray(OFDM_symbols), axis=0)
    T_guard = int(T_guard)
    return np.concatenate([t[t.shape[0] - T_guard:, :], t], axis=0)


def OFDM_demodulator(OFDM_time_guarded, T_guard):
    """`Task 5/OFDM_demodulator.m:2-9`: strip CP + column FFT (unscaled)."""
    x = np.asarray(OFDM_time_guarded)
    return np.fft.fft(x[int(T_guard):, :], axis=0)


def get_payload(RX_OFDM_symbols, dataCarriers):
    """`Task 5/get_payload.m:2-4`."""
    return np.asarray(RX_OFDM_symbols)[np.asarray(dataCarriers, dtype=np.int64) - 1, :]


# --------------------------------------------------------------------------- a10-a13
def add_STO(y, nSTO):
    """`Task 5/add_STO.m:1-10`."""
    y = np.asarray(y).ravel()
    n = int(nSTO)
    if n >= 0:
        return np.concatenate([y[n:], np.zeros(n, dtype=y.dtype)])
    return np.concatenate([np.zeros(-n, dtype=y.dtype), y[: y.size + n]])


def add_CFO(y, CFO, Nfft):
    """`Task 5/add_CFO.m:1-8`: phase ramp over the whole serial stream."""
    y = np.asarray(y).ravel()
    nn = np.arange(y.size, dtype=np.float64)
    return y * np.exp(2j * np.pi * CFO * nn / Nfft)


def Noise(SNR, IQ_TX, normals=None, rng=None):
    """`Task 5/Noise.m:1-12` -> (IQ_RX, N_var).  MATLAB draws the real block first and the
    imaginary block second (two ``normrnd`` calls, :7-8).  ``normals`` = (2, L) unit normals
    imports a shared realisation; otherwise ``rng`` (NumPy Generator) draws them in that order."""
    x = np.asarray(IQ_TX).ravel()
    P = np.mean(np.abs(x) ** 2)
    NoisePower = P / (10 ** (SNR / 10))
    if normals is None:
        rng = rng or np.random.default_rng()
        normals = np.stack([rng.standard_normal(x.size), rng.standard_normal(x.size)])
    normals = np.asarray(normals, dtype=np.float64)
    noise = np.sqrt(NoisePower / 2) * normals[0] + 1j * np.sqrt(NoisePower / 2) * normals[1]
    return x + noise, np.sqrt(NoisePower)


def get_MP_channel_resp(channel_taps, Nfft):
    """`Task 5/get_MP_channel_resp.m:2-19` -> (impulse_response, frequency_response)."""
    taps = np.asarray(channel_taps, dtype=np.float64).reshape(-1, 2)
    max_delay = int(taps[:, 0].max())
    h = np.zeros(max_delay + 1, dtype=np.float64)
    for delay, amp in taps:
        h[int(delay)] = amp                                      # :14 later rows overwrite
    return h, np.fft.fft(h, int(Nfft))


def apply_channel(x, h):
    """Script glue `Task 5/Main_model_Task_5.m:126-127`: ``conv(x,h,'full')`` truncated to len(x)."""
    x = np.asarray(x).ravel()
    h = np.asarray(h).ravel()
    return np.convolve(x, h, mode="full")[: x.size]


# --------------------------------------------------------------------------- a14-a16
def AutoCorrFunction(RxSignal, WidthWindow, Nfft):
    """`Task 5/AutoCorrFunction.m:1-28` -> (AutoCorr, TgPosition (1-based), FreqOffset).
    Windows are summed directly (not slid) so this is the exact-arithmetic definition."""
    r = np.asarray(RxSignal).ravel().astype(np.complex128)
    W = int(WidthWindow)
    Nfft = int(Nfft)
    n_out = r.size - W - Nfft
    prod = r[: r.size - Nfft] * np.conj(r[Nfft:])
    pw = np.abs(r) ** 2
    win = np.lib.stride_tricks.sliding_window_view
    num = win(prod, W)[:n_out].sum(axis=1)
    p1 = win(pw[: r.size - Nfft], W)[:n_out].sum(axis=1)
    p2 = win(pw[Nfft:], W)[:n_out].sum(axis=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        ac = num / np.sqrt(p1 * p2)                              # :5-6 (0/0 -> NaN)
    amp = np.abs(ac)
    with np.errstate(invalid="ignore"):
        idxs = np.nonzero(amp > 0.77)[0] + 1                     # :12 (1-based)
    idxs = idxs[idxs > W]                                        # :13
    tg = 65                                                      # :23 fallback
    if idxs.size:
        mask = np.concatenate([[True], np.abs(np.diff(idxs)) != 1])  # :15-16
        result = np.nonzero(mask)[0]                             # 0-based starts of runs
        if result.size >= 2:
            tg = int(np.floor((idxs[result[0]] + idxs[result[1] - 1]) / 2))  # :20
    freq = -np.angle(ac[tg - 1]) / (2 * np.pi)                   # :27
    return ac, tg, freq


def remove_IFO(rx_signal, Nfft):
    """`Task 5/remove_IFO.m:1-11`: first spectrum bin above 0.77 of the fixed window
    ``rx(Nfft+1:2*Nfft)``; raises IndexError like MATLAB when nothing crosses."""
    rx = np.asarray(rx_signal).ravel()
    Nfft = int(Nfft)
    spectrum = np.abs(np.fft.fft(rx[Nfft: 2 * Nfft]))
    inds = np.nonzero(spectrum > 0.77)[0]
    if inds.size == 0:
        raise IndexError("remove_IFO: no spectrum bin above 0.77 (inds(1) on empty)")
    IFO = int(inds[0])                                           # :8 (inds(1)-1, 0-based already)
    return add_CFO(rx, -IFO, Nfft), IFO


def fine_sync(rx_signal, pilotCarriers, pilotValues, time_desync, freq_desync, return_estimates=False):
    """`Task 4/fine_sync.m:1-60` (Task-4 mask: ``abs(diffs)<1e-3 & abs(diffs)~=0``).
    ``nn = 0:1023`` is hard-coded, so ``rx_signal`` must have 1024 rows when time_desync."""
    rx = np.array(rx_signal, dtype=np.complex128)
    pc = np.asarray(pilotCarriers, dtype=np.int64)
    tx = np.asarray(pilotValues).reshape(pc.size, -1)
    rxp = rx[pc - 1, :]
    deltak = float(pc[1] - pc[0])                                # :6
    txf = tx.ravel(order="F")
    q = txf * np.conj(rxp.ravel(order="F"))                      # :26-27
    taus = np.angle(q[1:] * np.conj(q[:-1])) / (2 * np.pi * deltak)  # :29
    diffs = np.diff(taus)                                        # :32
    mask = np.concatenate([[False], (np.abs(diffs) < 1e-3) & (np.abs(diffs) != 0)])  # :33
    taus_result = taus[mask]
    tail = taus_result[pc.size:]                                 # :35 (length(pilotCarriers)+1:end)
    tau = np.mean(tail) if tail.size else np.nan
    if time_desync:
        nn = np.arange(1024, dtype=np.float64)                   # :39
        nn_exp = np.exp(-2j * np.pi * tau * nn)
        rx = rx * np.conj(nn_exp)[:, None]                       # :42 nn_exp' = ctranspose
    rxp = rx[pc - 1, :]                                          # :47
    qks = np.angle(txf * np.conj(rxp.ravel(order="F")))          # :50
    sel = qks[np.abs(qks) > 1e-3]
    phase_shift = np.mean(sel) if sel.size else np.nan           # :52
    out = rx * np.exp(1j * phase_shift) if freq_desync else rx   # :54-58
    if return_estimates:
        return out, tau, phase_shift
    return out


# --------------------------------------------------------------------------- interp
def interp1_spline(x, y, xq):
    """MATLAB ``interp1(x,y,xq,'spline')``: not-a-knot cubic spline with extrapolation
    (2 points -> line, 3 points -> parabola), same as SciPy's ``CubicSpline(bc_type='not-a-knot')``."""
    x = np.asarray(x, dtype=np.float64).ravel()
    y = np.asarray(y).ravel()
    xq = np.asarray(xq, dtype=np.float64)
    if x.size == 2:
        return y[0] + (y[1] - y[0]) * (xq - x[0]) / (x[1] - x[0])
    if not np.all(np.isfinite(y)):          # MATLAB propagates NaN through the spline; SciPy refuses it
        return np.full(xq.shape, np.nan + 1j * np.nan if np.iscomplexobj(y) else np.nan)
    cs = CubicSpline(x, y, bc_type="not-a-knot", extrapolate=True)
    return cs(xq)


def interpolate(H, pilot_loc, Nfft, method):
    """`Task 5/interpolate.m:1-24` (third argument is the output length, N_carrier as called)."""
    H = np.asarray(H).ravel().astype(np.complex128)
    loc = np.asarray(pilot_loc, dtype=np.float64).ravel()
    N = int(Nfft)
    if loc[0] > 1:                                               # :7-10
        slope = (H[1] - H[0]) / (loc[1] - loc[0])
        H = np.concatenate([[H[0] - slope * (loc[0] - 1)], H])
        loc = np.concatenate([[1.0], loc])
    if loc[-1] < N:                                              # :12-16
        slope = (H[-1] - H[-2]) / (loc[-1] - loc[-2])
        H = np.concatenate([H, [H[-1] + slope * (N - loc[-1])]])
        loc = np.concatenate([loc, [float(N)]])
    xq = np.arange(1, N + 1, dtype=np.float64)
    if str(method)[0].lower() == "l":                            # :18-19
        return np.interp(xq, loc, H.real) + 1j * np.interp(xq, loc, H.imag)
    return interp1_spline(loc, H, xq)                            # :21


# --------------------------------------------------------------------------- a17-a21
def estimate_channel(rx_signal, allCarriers, pilotCarriers, pilotValues):
    """`Task 5/estimate_channel.m:1-10` -> (H_est over allCarriers, Hest_at_pilots)."""
    pc = np.asarray(pilotCarriers, dtype=np.int64)
    rxp = np.asarray(rx_signal)[pc - 1, :]
    tx = np.asarray(pilotValues).reshape(pc.size, -1)
    Hp = np.mean(rxp / tx, axis=1)                               # :6
    return interp1_spline(pc, Hp, np.asarray(allCarriers, dtype=np.float64)), Hp


def LS_CE(Y, Xp, pilot_loc, N_carrier):
    """`Task 5/LS_CE.m:1-34`: linear indexing => first symbol column only (:27-28)."""
    loc = np.asarray(pilot_loc, dtype=np.int64).ravel()
    Yf = np.asarray(Y).ravel(order="F")
    Xf = np.asarray(Xp).ravel(order="F")
    LS_est = Yf[loc - 1] / Xf[: loc.size]
    return interpolate(LS_est, loc, N_carrier, "spline")


def MMSE_CE(Y, Xp, pilot_loc, Nfft, N_carrier, h, SNR):
    """`Task 5/MMSE_CE.m:1-39` (dense restatement, including the discarded rows of Rhp)."""
    snr = 10 ** (SNR * 0.1)
    loc = np.asarray(pilot_loc, dtype=np.int64).ravel()
    Np = loc.size
    Nps = float(loc[1] - loc[0])                                 # :15
    Y = np.asarray(Y)
    Xp = np.asarray(Xp).reshape(Np, -1)
    H_tilde = Y[loc - 1, 0] / Xp[:, 0]                           # :17
    h = np.asarray(h).ravel().astype(np.complex128)
    k = np.arange(h.size, dtype=np.float64)                      # :19
    hh = np.vdot(h, h)                                           # h*h'
    tmp = h * np.conj(h) * k
    r = np.sum(tmp) / hh
    r2 = (tmp @ k) / hh
    tau_rms = np.sqrt(r2 - r ** 2)                               # :24
    df = 1.0 / N_carrier
    j2pi_tau_df = 1j * 2 * np.pi * tau_rms * df                  # :26
    K1 = np.arange(N_carrier, dtype=np.float64)[:, None]
    K2 = np.arange(Np, dtype=np.float64)[None, :]
    rf = 1.0 / (1 + j2pi_tau_df * Nps * (K1 - K2))               # :30
    K3 = np.arange(Np, dtype=np.float64)[:, None]
    rf2 = 1.0 / (1 + j2pi_tau_df * Nps * (K3 - K2))              # :33
    Rpp = rf2 + np.eye(Np) / snr                                 # :35
    H = rf @ np.linalg.solve(Rpp, H_tilde)                       # :36  (Rhp/Rpp)*H_tilde.'
    return interpolate(H[:Np], loc, N_carrier, "spline")        # :38


def equalize_signal(OFDM_demod, Hest, N_carrier):
    """`Task 5/equalize_signal.m:1-8`: one-tap ZF on rows 1:N_carrier, zeros elsewhere."""
    X = np.asarray(OFDM_demod)
    out = np.zeros(X.shape, dtype=np.complex128)
    Hest = np.asarray(Hest).ravel()
    with np.errstate(divide="ignore", invalid="ignore"):
        out[:N_carrier, :] = X[:N_carrier, :] / Hest[:N_carrier, None]
    return out


# --------------------------------------------------------------------------- a22/a23
def sensing_matrix_dft(pilotCarriers, Nfft, Ldict):
    """Script glue `Task 5/Main_model_Task_5.m:182-190`: ``P*dftmtx(Nfft)(:,1:Ldict)`` i.e.
    ``A(i,l) = exp(-2*pi*1j*(p_i-1)*(l-1)/Nfft)``."""
    p = np.asarray(pilotCarriers, dtype=np.int64).ravel() - 1
    l = np.arange(int(Ldict), dtype=np.int64)
    ph = (p[:, None] * l[None, :]) % int(Nfft)
    return np.exp(-2j * np.pi * ph / Nfft)


def OMP_estimate(Y, sensing_matrix, Nfft, dominant_taps, SNR_dB=None):
    """`Task 5/OMP_estimate.m:2-37` -> (H_OMP (Nfft,), h_impulse_est (Nfft,), index (1-based))."""
    A_full = np.asarray(sensing_matrix, dtype=np.complex128)
    y = np.asarray(Y).ravel().astype(np.complex128)
    index = [int(np.argmax(np.abs(A_full.conj().T @ y))) + 1]   # :7
    A = A_full[:, [index[0] - 1]]
    x = np.linalg.pinv(A) @ y                                    # :9
    residue = [y - A @ x]                                        # :11
    for _ in range(2, int(dominant_taps) + 1):                   # :13
        index.append(int(np.argmax(np.abs(A_full.conj().T @ residue[-1]))) + 1)
        A = np.concatenate([A, A_full[:, [index[-1] - 1]]], axis=1)
        x = np.linalg.pinv(A) @ y                                # :17 re-solve on the measurement
        residue.append(y - A @ x)
        if np.linalg.norm(residue[-1] - residue[-2]) / np.linalg.norm(residue[-2]) < 1e-2:  # :20
            break
    h = np.zeros(int(Nfft), dtype=np.complex128)
    for i1, idx in enumerate(index):                             # :31-33 later duplicates overwrite
        h[idx - 1] = x[i1]
    return np.fft.fft(h), h, np.array(index, dtype=np.int64)


def MP_estimate(Y, sensing_matrix, Nfft, dominant_taps):
    """`Task 5/MP_estimate.m:2-34` -> (H_MP (Nfft,), h_impulse_est (Nfft,)).  Only the first
    ``Np = size(sensing_matrix,1)`` dictionary columns are searched (:3,10)."""
    A = np.asarray(sensing_matrix, dtype=np.complex128)
    Np = A.shape[0]
    residue = np.asarray(Y).ravel().astype(np.complex128).copy()
    K = int(dominant_taps)
    kp = np.zeros(K, dtype=np.int64)
    x = np.zeros(K, dtype=np.complex128)
    norms2 = np.sum(np.abs(A[:, :Np]) ** 2, axis=0)
    for i1 in range(K):
        proj = np.abs(A[:, :Np].conj().T @ residue) ** 2 / norms2   # :15
        picked = kp[kp > 0] - 1
        proj[picked] = -100.0                                    # :11-12
        kp[i1] = int(np.argmax(proj)) + 1                        # :18
        a = A[:, kp[i1] - 1]
        x[i1] = np.vdot(a, residue) / norms2[kp[i1] - 1]         # :22
        residue = residue - a * x[i1]                            # :21,23
    h = np.zeros(int(Nfft), dtype=np.complex128)
    for i1 in range(K):
        h[kp[i1] - 1] = x[i1]                                    # :28-30
    return np.fft.fft(h), h


# --------------------------------------------------------------------------- a24/a25
def BER_func(Bit_Tx, Bit_Rx):
    """`Task 5/BER_func.m:1-7`."""
    tx = np.asarray(Bit_Tx).ravel()
    rx = np.asarray(Bit_Rx).ravel()
    return float(np.sum(tx != rx)) / tx.size


def MER_func(IQ_RX, Constellation, return_sums=False):
    """`Task 5/MER_func.m:1-26`: nearest point by ``abs`` with strict ``<`` (first min)."""
    d, _ = constellation_func(Constellation)
    rx = np.asarray(IQ_RX).ravel()
    dist = np.abs(rx[None, :] - d[:, None])
    ideal = d[np.argmin(dist, axis=0)]
    sum1 = np.sum(ideal.real ** 2 + ideal.imag ** 2)
    e = ideal - rx
    sum2 = np.sum(e.real ** 2 + e.imag ** 2)
    with np.errstate(divide="ignore"):
        mer = 10 * np.log10(sum1 / sum2)
    return (mer, sum1, sum2) if return_sums else mer


# --------------------------------------------------------------------------- glue
def pilot_layout_percent(N_carrier, percent, Nfft, last_gap):
    """Pilot/data index construction of Tasks 1-4 (`Task 4/Main_model_Task_4.m:14-24`):
    ``pilots = [1:step:N_carrier-last_gap, N_carrier]``; ``last_gap`` is 2 in Tasks 1-4 and 1
    in the comb==1 branch of Task 5 (`Task 5/Main_model_Task_5.m:28-31`)."""
    amount = int(np.floor(percent / 100 * N_carrier + 0.5))      # MATLAB round (half away from 0)
    step = N_carrier // amount
    pilots = np.concatenate([np.arange(1, N_carrier - last_gap + 1, step), [N_carrier]])
    pilots = np.unique(pilots)
    data = np.setdiff1d(np.arange(1, N_carrier + 1), pilots)
    return pilots.astype(np.int64), data.astype(np.int64)


def pilot_layout_comb(N_carrier, comb):
    """`Task 5/Main_model_Task_5.m:18-22,34`: ``pilots = 1:comb:N_carrier``."""
    pilots = np.arange(1, N_carrier + 1, int(comb))
    data = np.setdiff1d(np.arange(1, N_carrier + 1), pilots)
    return pilots.astype(np.int64), data.astype(np.int64)


def calculatePAPR(OFDM_signal):
    """`Task 5/calculatePAPR.m:2-11`."""
    a = np.abs(np.asarray(OFDM_signal).ravel())
    return 10 * np.log10(a.max() ** 2 / np.mean(a ** 2))


def calculate_window_PAPR(Tx_OFDM_Signal, Nfft):
    """`Task 5/calculate_window_PAPR.m:2-15` (direct O(L*Nfft) definition)."""
    p = np.abs(np.asarray(Tx_OFDM_Signal).ravel()) ** 2
    w = np.lib.stride_tricks.sliding_window_view(p, int(Nfft))
    return 10 * np.log10(w.max(axis=1) / w.mean(axis=1))


def calculateCCDF(PAPR_values):
    """`Task 5/calculateCCDF.m:2-6` -- ``ecdf`` then complement; returns (x, CCDF) with the
    MATLAB ``ecdf`` convention of a leading duplicate of the smallest x with F = 0."""
    v = np.sort(np.asarray(PAPR_values).ravel())
    x, counts = np.unique(v, return_counts=True)
    F = np.cumsum(counts) / v.size
    x = np.concatenate([[x[0]], x])
    F = np.concatenate([[0.0], F])
    return x, 1 - F
