"""Script-level glue of the reference, restated (test infrastructure; PARITY UNPINNED, see
``oracle/__init__.py``).  Each chain composes the per-function oracle in the order the
reference scripts call it, for ONE serial stream (``N_symb`` OFDM symbols); batches are
Python loops over streams.  Citations are ``path:line`` under ``/root/reference/``.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import functions as F


@dataclass
class LinkParams:
    """Literals at the top of the reference scripts (`Task 5/Main_model_Task_5.m:6-46`)."""
    Nfft: int = 4096
    N_carrier: int = 1024
    T_Guard: int = 512
    Amount_OFDM_Frames: int = 2
    Amount_ODFM_SpF: int = 7
    Constellation: str = "16QAM"
    pilotCarriers: np.ndarray = field(default=None)      # 1-based
    dataCarriers: np.ndarray = field(default=None)       # 1-based
    pilotValues: np.ndarray = field(default=None)        # (Np, N_symb)
    Register: np.ndarray = field(default_factory=lambda: F.DEFAULT_REGISTER.copy())

    @property
    def N_symb(self):
        return self.Amount_OFDM_Frames * self.Amount_ODFM_SpF

    @property
    def bps(self):
        return F.constellation_func(self.Constellation)[1]

    @property
    def frame_bits(self):
        return self.Amount_ODFM_SpF * len(self.dataCarriers) * self.bps

    @property
    def stream_bits(self):
        return self.frame_bits * self.Amount_OFDM_Frames

    @property
    def stream_len(self):
        return self.N_symb * (self.Nfft + self.T_Guard)


def make_pilot_values(Np, N_symb, Constellation, scale, alternate):
    """`Task 4/Main_model_Task_4.m:31-36` / `Task 5/Task5_part2.m:85-91`: amplitude
    ``scale*max|dict|``; ``exp(1i*pi)`` and the ctranspose in ``repmat(pilotValues',...)`` are
    kept, so "-a" carries an imaginary part of about -a*1.2e-16."""
    d, _ = F.constellation_func(Constellation)
    amp = scale * np.max(np.abs(d))
    pv = np.zeros(Np, dtype=np.complex128)
    pv[:] = amp * np.exp(1j * 0)
    if alternate:
        pv[1::2] = amp * np.exp(1j * np.pi)
    return np.tile(np.conj(pv)[:, None], (1, N_symb)), amp


def params_task5(comb=4, scale=2.0, alternate=True):
    """M1 / Task-5 part-2 shape (`Task 5/Task5_part2.m:5-17,46-91`)."""
    p = LinkParams()
    p.pilotCarriers, p.dataCarriers = F.pilot_layout_comb(p.N_carrier, comb)
    p.pilotValues, _ = make_pilot_values(len(p.pilotCarriers), p.N_symb, p.Constellation, scale, alternate)
    return p


def params_task4(percent=15, scale=4.0 / 3.0, alternate=True, Constellation="16QAM"):
    """Task-4 shape (`Task 4/Main_model_Task_4.m:6-36`)."""
    p = LinkParams(Nfft=1024, N_carrier=400, T_Guard=128, Amount_OFDM_Frames=10, Amount_ODFM_SpF=5,
                   Constellation=Constellation)
    p.pilotCarriers, p.dataCarriers = F.pilot_layout_percent(p.N_carrier, percent, p.Nfft, last_gap=2)
    p.pilotValues, _ = make_pilot_values(len(p.pilotCarriers), p.N_symb, p.Constellation, scale, alternate)
    return p


def scramble_frames(p: LinkParams, bits, descramble=False, fast=False):
    """Per-frame register reset (`Task 4/Main_model_Task_4.m:43-58`, `:350-364`).  ``fast`` selects the
    vectorised (bit-identical) forms, used only where the oracle is timed as the CPU baseline."""
    if fast:
        fn = F.DeScrambler_fast if descramble else F.Scrambler_fast
    else:
        fn = F.DeScrambler if descramble else F.Scrambler
    L = p.frame_bits
    out = np.empty(p.stream_bits, dtype=np.uint8)
    for i in range(p.Amount_OFDM_Frames):
        out[i * L:(i + 1) * L], _ = fn(p.Register, bits[i * L:(i + 1) * L])
    return out


def tx_chain(p: LinkParams, input_bits, scramble=True, fast=False):
    """bits -> Scrambler -> mapping -> OFDM_map_carriers -> OFDM_modulator -> serial stream
    (`Task 5/Main_model_Task_5.m:53-85`).  Returns (stream, grid, sc_bits)."""
    bits = np.asarray(input_bits).ravel()
    sc = scramble_frames(p, bits, fast=fast) if scramble else bits.astype(np.uint8)
    iq, pad = F.mapping(sc, p.Constellation)
    grid = F.OFDM_map_carriers(iq, p.N_symb, p.Nfft, p.dataCarriers, p.pilotCarriers, p.pilotValues)
    tx = F.OFDM_modulator(grid, p.T_Guard)
    return tx.ravel(order="F"), grid, sc


def channel_task5(p: LinkParams, tx, SNR_dB, taps, normals=None, rng=None):
    """Noise first, then multipath (`Task 5/Main_model_Task_5.m:108,123-127`)."""
    rx = tx
    if SNR_dB is not None:
        rx, _ = F.Noise(SNR_dB, rx, normals=normals, rng=rng)
    if taps is not None:
        h, _ = F.get_MP_channel_resp(taps, p.Nfft)
        rx = F.apply_channel(rx, h)
    return rx


def rx_chain_task5(p: LinkParams, rx_stream, input_bits, descramble=True, method="LS", h_true=None, SNR_dB=None, fast=False):
    """M1 chain: OFDM_demodulator -> LS_CE -> equalize_signal -> get_payload -> demapping ->
    DeScrambler -> BER_func (`Task 5/Task5_part2.m:169-174,269-303`, per-frame descrambler
    reset as `Task 5/Main_model_Task_5.m:262-271`).  Returns dict."""
    X = np.asarray(rx_stream).reshape((p.Nfft + p.T_Guard, p.N_symb), order="F")
    Y = F.OFDM_demodulator(X, p.T_Guard)
    if method == "LS":
        H = F.LS_CE(Y, p.pilotValues, p.pilotCarriers, p.N_carrier)
    elif method == "MMSE":
        h = h_true if h_true is not None else np.fft.ifft(F.LS_CE(Y, p.pilotValues, p.pilotCarriers, p.N_carrier))
        H = F.MMSE_CE(Y, p.pilotValues, p.pilotCarriers, p.Nfft, p.N_carrier, h, SNR_dB)
    else:
        raise ValueError(method)
    eq = F.equalize_signal(Y, H, p.N_carrier)
    rx_iq = F.get_payload(eq, p.dataCarriers).ravel(order="F")
    out_bits = F.demapping(-1, rx_iq, p.Constellation)
    dsc = scramble_frames(p, out_bits, descramble=True, fast=fast) if descramble else out_bits
    tx_bits = np.asarray(input_bits).ravel()
    n_err = int(np.sum(tx_bits != dsc))
    return {"Y": Y, "H": H, "eq": eq, "rx_iq": rx_iq, "bits": dsc, "raw_bits": out_bits,
            "errors": n_err, "n_bits": tx_bits.size}


def impair_task4(p: LinkParams, tx, SNR_dB=None, Time_Delay=None, Freq_Shift=None, taps=None, normals=None, rng=None):
    """Impairments in Task-4 order: Noise -> add_STO -> add_CFO -> multipath
    (`Task 4/Main_model_Task_4.m:95,103,110,263-264`)."""
    rx = np.asarray(tx)
    if SNR_dB is not None:
        rx, _ = F.Noise(SNR_dB, rx, normals=normals, rng=rng)
    if Time_Delay is not None:
        rx = F.add_STO(rx, Time_Delay)
    if Freq_Shift is not None:
        rx = F.add_CFO(rx, Freq_Shift, p.Nfft)
    if taps is not None:
        h, _ = F.get_MP_channel_resp(taps, p.Nfft)
        rx = F.apply_channel(rx, h)
    return rx


def rx_chain_task4(p: LinkParams, rx_stream, input_bits, time_desync=True, freq_desync=True, mp_desync=True, descramble=True,
                   ifo_passthrough=False):
    """M2 chain (`Task 4/Main_model_Task_4.m:277-366`): AutoCorrFunction -> add_STO x2 -> add_CFO ->
    remove_IFO -> reshape -> OFDM_demodulator -> fine_sync -> estimate_channel -> equalize_signal ->
    get_payload -> demapping -> DeScrambler -> BER.  remove_IFO raises like MATLAB when no spectrum bin
    exceeds 0.77; with ``ifo_passthrough`` the stream passes unchanged with IFO = -1 instead, as the
    device library does (`ofdm_remove_ifo`).  ``raw_bits`` are the decisions before DeScrambler."""
    rx = np.asarray(rx_stream).ravel()
    info = {}
    if time_desync or freq_desync:
        ac, tg, fo = F.AutoCorrFunction(rx, p.T_Guard, p.Nfft)
        info.update(TgPosition=tg, FreqOffset=fo)
        if time_desync:
            rx = F.add_STO(rx, tg)
            rx = F.add_STO(rx, -(p.Nfft + p.T_Guard))
    if freq_desync:
        rx = F.add_CFO(rx, -fo, p.Nfft)
        try:
            rx, ifo = F.remove_IFO(rx, p.Nfft)
        except IndexError:
            if not ifo_passthrough:
                raise
            ifo = -1
        info.update(IFO=ifo)
    X = rx.reshape((p.Nfft + p.T_Guard, p.N_symb), order="F")
    Y = F.OFDM_demodulator(X, p.T_Guard)
    if time_desync or freq_desync:
        Y, tau, ph = F.fine_sync(Y, p.pilotCarriers, p.pilotValues, time_desync, freq_desync, return_estimates=True)
        info.update(tau=tau, phase_shift=ph)
    if mp_desync:
        H, Hp = F.estimate_channel(Y, np.arange(1, p.Nfft + 1), p.pilotCarriers, p.pilotValues)
        info.update(H=H)
        Y = F.equalize_signal(Y, H, p.N_carrier)
    rx_iq = F.get_payload(Y, p.dataCarriers).ravel(order="F")
    out_bits = F.demapping(-1, rx_iq, p.Constellation)
    dsc = scramble_frames(p, out_bits, descramble=True) if descramble else out_bits
    tx_bits = np.asarray(input_bits).ravel()
    info.update(Y=Y, rx_iq=rx_iq, bits=dsc, raw_bits=out_bits, errors=int(np.sum(tx_bits != dsc)), n_bits=tx_bits.size)
    return info


def read_payload_bits(tiff_path, size_buffer):
    """`Task 5/file_reader.m:2-12`: ``imbinarize`` = Otsu threshold on the 256-bin histogram,
    column-major flatten, truncate."""
    from PIL import Image
    img = np.asarray(Image.open(tiff_path)).astype(np.float64)
    counts = np.bincount(img.astype(np.int64).ravel(), minlength=256).astype(np.float64)
    p = counts / counts.sum()
    omega = np.cumsum(p)
    mu = np.cumsum(p * np.arange(1, 257))
    mu_t = mu[-1]
    with np.errstate(divide="ignore", invalid="ignore"):
        sigma_b2 = (mu_t * omega - mu) ** 2 / (omega * (1 - omega))
    sigma_b2[~np.isfinite(sigma_b2)] = -np.inf
    mx = sigma_b2.max()
    level = (np.mean(np.nonzero(sigma_b2 == mx)[0]) ) / 255.0     # graythresh: mean of maxima, (idx-1)/(nbins-1)
    bw = (img / 255.0) > level
    return bw.ravel(order="F")[:size_buffer].astype(np.uint8)


# ---------------------------------------------------------------------------------------------------------
# Task 5 part 2: comb sweep x Monte-Carlo runs x four estimators (`Task 5/Task5_part2.m`)

def part2_combs(N_carrier=1024, lo=4, hi=256):
    """`combs = 4:1:256` de-duplicated by floor(N_carrier/comb), first comb of each pilot count kept
    (`Task5_part2.m:13-17`: unique() returns first occurrences, ascending in the value)."""
    combs = np.arange(lo, hi + 1)
    amounts = N_carrier // combs
    _, ia = np.unique(amounts, return_index=True)
    combs = combs[np.sort(ia)]
    return combs, N_carrier // combs


def params_part2(comb=None, pilotCarriers=None):
    """Pilot layout and values of one sweep point (`Task5_part2.m:46-91`): regular comb `1:comb:N_carrier` or
    a given sorted random mask (`sort(randperm(1024, Np))`, `:57-65`); alternating +-2*max|dict| pilots."""
    p = LinkParams()
    if pilotCarriers is None:
        p.pilotCarriers, p.dataCarriers = F.pilot_layout_comb(p.N_carrier, comb)
    else:
        p.pilotCarriers = np.asarray(pilotCarriers, dtype=np.int64)
        allc = np.arange(1, p.N_carrier + 1)
        p.dataCarriers = allc[~np.isin(allc, p.pilotCarriers)]
    p.pilotValues, _ = make_pilot_values(len(p.pilotCarriers), p.N_symb, p.Constellation, 2.0, True)
    return p


# 3GPP TS 36.101 Annex B.2.1 (the delay profiles `lteFadingChannel` implements; `Task5_part2.m:29`): ns, dB
TDL_PROFILES = {
    "EPA": ([0, 30, 70, 90, 110, 190, 410], [0.0, -1.0, -2.0, -3.0, -8.0, -17.2, -20.8]),
    "EVA": ([0, 30, 150, 310, 370, 710, 1090, 1730, 2510], [0.0, -1.5, -1.4, -3.6, -0.6, -9.1, -7.0, -12.0, -16.9]),
    "ETU": ([0, 50, 120, 200, 230, 500, 1600, 2300, 5000], [-1.0, -1.0, -1.0, 0.0, 0.0, 0.0, -3.0, -5.0, -7.0]),
}
TDL_LEAD = 7


def tdl_amplitudes(profile):
    """Tap amplitudes normalised to unit total average power (lteFadingChannel's NormalizePathGains default)."""
    pw = 10.0 ** (np.asarray(TDL_PROFILES[profile][1]) / 10.0)
    return np.sqrt(pw / pw.sum())


def tdl_impulse_response(profile, fs_hz, path_gains):
    """Impulse response of the static tapped-delay-line model for given complex path gains (the analogue of
    `info.PathGains`, amplitudes included): Hann-windowed sinc interpolation of the fractional delays with a
    lead of TDL_LEAD samples.  lteFadingChannel's own interpolator is not public -- this is the published
    model only (PARITY UNPINNED against MATLAB)."""
    d = np.asarray(TDL_PROFILES[profile][0], dtype=np.float64) * 1e-9 * fs_hz
    n = np.arange(int(np.ceil(d.max())) + 2 * TDL_LEAD + 1, dtype=np.float64)
    x = n[None, :] - TDL_LEAD - d[:, None]
    w = np.where(np.abs(x) < TDL_LEAD, np.sinc(x) * (0.5 + 0.5 * np.cos(np.pi * x / TDL_LEAD)), 0.0)
    return (np.asarray(path_gains)[:, None] * w).sum(axis=0)


def part2_run(p: LinkParams, tx_noised, h_t, input_bits, n_paths, SNR_dB, Ldict):
    """One Monte-Carlo run (`Task5_part2.m:148-304`) for a given static impulse response `h_t` (what
    `lteFadingChannel(local_channel,[1; zeros(Nfft-1,1)])` returns, `:154`).  Returns NMSE[4], errors[4]
    in the script's order LS, MMSE, MP, OMP."""
    Nc = p.N_carrier
    h_full = np.zeros(p.Nfft, dtype=np.complex128)
    h_full[: len(h_t)] = h_t
    rx = F.apply_channel(np.asarray(tx_noised), np.asarray(h_t))                           # :152 (filtering, first L samples)
    H_f = np.fft.fft(h_full)                                                               # :155
    X = rx.reshape((p.Nfft + p.T_Guard, p.N_symb), order="F")                              # :169
    Y = F.OFDM_demodulator(X, p.T_Guard)                                                   # :172
    H_ls = F.LS_CE(Y, p.pilotValues, p.pilotCarriers, Nc)                                  # :174
    H_mmse = F.MMSE_CE(Y, p.pilotValues, p.pilotCarriers, p.Nfft, Nc, h_full[:Nc], SNR_dB)  # :176-177
    A = F.sensing_matrix_dft(p.pilotCarriers, p.Nfft, Ldict)                               # :181-189
    Yp = Y[p.pilotCarriers - 1, 0] / p.pilotValues[:, 0]                                   # :190
    H_mp, _ = F.MP_estimate(Yp, A, p.Nfft, n_paths)                                        # :192
    H_omp, _, _ = F.OMP_estimate(Yp, A, p.Nfft, n_paths, SNR_dB)                           # :193
    ests = [H_ls, H_mmse, np.asarray(H_mp).ravel(), np.asarray(H_omp).ravel()]
    nmse, errs = [], []
    tx_bits = np.asarray(input_bits).ravel()
    for H in ests:
        e = H_f[:Nc] - np.asarray(H).ravel()[:Nc]
        nmse.append(float(np.real(np.vdot(e, e))) / Nc)                                    # :200-203
        eq = F.equalize_signal(Y, np.asarray(H).ravel(), Nc)                               # :269-272
        rx_iq = F.get_payload(eq, p.dataCarriers).ravel(order="F")                         # :279-280
        out_bits = F.demapping(-1, rx_iq, p.Constellation)                                 # :283
        errs.append(int(np.sum(tx_bits != out_bits)))                                      # :303
    return np.asarray(nmse), np.asarray(errs), {"H_f": H_f, "H": ests, "Y": Y}
