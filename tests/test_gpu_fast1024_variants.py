"""Every instantiation of the Nfft-1024 Task-4 receiver -- the fused persistent kernel (`rx_t4_fast_kernel<K2N, QAM16, NEAR>`),
the split chain for large batches (`t4_ifo_kernel` -> `t4_sym_kernel<K2N>` -> `t4_post_kernel<QAM16, NEAR, false>`) and the
fallbacks to the generic block-FFT kernel (`rx_t4_kernel`) -- and the Nfft-1024 transmitter (`tx1024_kernel`) against the float64
oracle (`OC.rx_chain_task4`, `OC.tx_chain`): both second-DFT widths (K2N = 13 for N_carrier <= 416, 32 above), every
constellation, descrambler frame geometries, stream lengths, guards, receiver stages, estimator corners, batch sizes around the
persistent grid and across the split chain's passes, and the optional outputs.

Which kernels ran is read from the CUDA activity of `torch.profiler` (tests/kernel_witness.py): the dispatch in
`ofdm_rx_chain_t4_ex` picks a kernel from the shared memory a stream shape needs, and a launch counter cannot tell them apart.
A box without CUPTI skips those asserts and still runs the parity ones."""
import ctypes as C

import numpy as np
import pytest

import oracle as O
from oracle import chains as OC
from kernel_witness import Registry, t4_phase_bounds, witness

pytestmark = pytest.mark.gpu
TAPS4 = [[0, 1], [4, .6], [10, .3]]
# a scrambler register with cells 13 and 14 set: both taps of the pre-history fold (`Scrambler.m:18-28`) are exercised
REG = np.array([1, 1, 0, 1, 0, 0, 1, 1, 1, 0, 0, 1, 1, 1, 1], dtype=np.uint8)
SNR_DB = 30.0
# Relative error of the FP32 equalised symbols against the oracle's.  The channel estimate is held to 1e-3 of the oracle's
# (relative, once exp(j dphi) is taken out); the phase estimate's own error dphi cancels in Y * cf / H when the equaliser runs
# (cf and H carry the same exp(j phase)) and rotates the symbols by dphi when it does not.  A symbol e moved by |de| changes
# its decision margin (second-smallest minus smallest squared distance) by at most 2 * D * |de|, D the constellation's
# diameter, and |de| <= R * (EQ_REL + [mp_desync off] * |dphi|), R the largest |e| of the stream: decisions may differ from
# the oracle's only where the float64 margin is below that bound (_slack).
EQ_REL = 1e-3
NEAR = 1e-3


@pytest.fixture(scope="module")
def G():
    import ofdm_b200
    return ofdm_b200


def rel_err(a, b):
    return np.linalg.norm((np.asarray(a) - np.asarray(b)).ravel()) / max(np.linalg.norm(np.asarray(b).ravel()), 1e-300)


def _lp(ctx, p, scramble=True):
    return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                           p.pilotCarriers, p.pilotValues, Register=p.Register, scramble=scramble)


def _link(Nc=400, S=10, SpF=5, pct=15, con="16QAM", Tg=128, Nfft=1024, reg=False, past=0):
    """Task-4 shape (`Main_model_Task_4.m:6-36`, percent-style layout, alternating pilots of 4/3 max|dictionary|); `past` data
    carriers N_carrier + 1 .. N_carrier + past are appended (they carry payload but no equaliser tap: decided from 0)."""
    p = OC.LinkParams(Nfft=Nfft, N_carrier=Nc, T_Guard=Tg, Amount_OFDM_Frames=S // SpF, Amount_ODFM_SpF=SpF, Constellation=con)
    p.pilotCarriers, p.dataCarriers = O.pilot_layout_percent(Nc, pct, Nfft, last_gap=2)
    if past:
        p.dataCarriers = np.concatenate([p.dataCarriers, np.arange(Nc + 1, Nc + past + 1)])
    p.pilotValues, _ = OC.make_pilot_values(len(p.pilotCarriers), p.N_symb, con, 4.0 / 3.0, True)
    if reg:
        p.Register = REG.copy()
    return p


def _detector_failed(rx, W, Nfft):
    """AutoCorrFunction found fewer than two runs above 0.77 and fell back to TgPosition = 65 (`AutoCorrFunction.m:21-24`)."""
    ac, _, _ = O.AutoCorrFunction(rx, W, Nfft)
    with np.errstate(invalid="ignore"):
        idx = np.nonzero(np.abs(ac) > 0.77)[0] + 1
    idx = idx[idx > W]
    return idx.size == 0 or not np.any(np.diff(idx) != 1)


# A stream: (STO, CFO) of impair_task4 at SNR_DB with TAPS4, optionally (STO, CFO, scale) -- the received samples times scale,
# which leaves every estimate but remove_IFO's threshold unchanged -- or "noise" (unit-power noise: the detector fails).
T4_STREAMS = [(37, 7.24), (900, 0.24), (150, 12.4), (0, 0.0), (611, 3.3), (1152, 30.4), (1, 0.49), (77, 21.7)]
DEFAULT = [(900, 0.24), (611, 3.3), (1, 0.49)]
FRACTIONAL = [(900, 0.24), (1, 0.49), (300, -0.3)]      # full-band layouts: an integer CFO puts data in the IFO search's first bins


def _make_streams(p, spec, seed, scramble=True, flags=(1, 1, 1)):
    """Payloads through the oracle's TX chain and the Task-4 impairments (multipath only when the receiver equalises), rounded
    to the FP32 samples the kernels read, and the oracle's receiver on each (with the same stages, descrambler and IFO
    pass-through the library has)."""
    rng = np.random.default_rng(seed)
    n = len(spec)
    bits = rng.integers(0, 2, (n, p.stream_bits)).astype(np.uint8)
    rxs, refs = [], []
    for b, s in enumerate(spec):
        if s == "noise":
            rx = (rng.standard_normal(p.stream_len) + 1j * rng.standard_normal(p.stream_len)) / np.sqrt(2)
        else:
            tx, _, _ = OC.tx_chain(p, bits[b], scramble=scramble, fast=True)
            rx = OC.impair_task4(p, tx, SNR_dB=SNR_DB, Time_Delay=s[0], Freq_Shift=s[1], taps=TAPS4 if flags[2] else None, rng=rng)
            if len(s) > 2:
                rx = rx * s[2]
        rx = rx.astype(np.complex64)
        rxs.append(rx)
        ref = OC.rx_chain_task4(p, rx.astype(np.complex128), bits[b], *flags, descramble=scramble, ifo_passthrough=True)
        if flags[0] or flags[1]:
            ref["fail"] = int(_detector_failed(rx.astype(np.complex128), p.T_Guard, p.Nfft))
        refs.append(ref)
    return bits, np.stack(rxs), refs


def _slack(p, ref, rot, mp):
    """Largest change of a decision margin the FP32 chain may cause on this stream (EQ_REL above); rot bounds the rotation
    the estimates' differences leave on the symbols when the equaliser does not cancel it."""
    d, _ = O.constellation_func(p.Constellation)
    D = np.max(np.abs(d[:, None] - d[None, :]))
    R = np.max(np.abs(ref["rx_iq"]))
    rot = 0.0 if mp or not np.isfinite(rot) else rot
    return 2 * D * R * (EQ_REL + rot)


def _tau_tol(p, rx, ref, td, fd):
    """fine_sync's tau (`fine_sync.m:25-35`) is the mean of the pilot-pair angles that pass the mask |diff| < 1e-3 & diff ~= 0,
    after the first Np of them.  Where add_STO zero-filled a symbol, the pair angle of an exact-zero pilot is 0 or +-pi by
    the signs of the zeros alone.  Two such values never pass the mask together (their differences are 0, 1/(12 dk) or
    1/(6 dk)), so only the A mask entries that compare one of them with a pilot-pair angle below 1e-3 depend on the signs.
    Each can add, drop or swap one term of the mean of n terms, all inside [lo, hi] (the kept values and 0): tau is fixed
    to 2 * A * (hi - lo) / (n - 2 * A) on top of FP32 rounding (2e-5)."""
    x = np.asarray(rx, dtype=np.complex128).ravel()
    if td:
        x = O.add_STO(O.add_STO(x, ref["TgPosition"]), -(p.Nfft + p.T_Guard))
    if fd:
        x = O.add_CFO(x, -ref["FreqOffset"], p.Nfft)
        if ref["IFO"] >= 0:
            x, _ = O.remove_IFO(x, p.Nfft)
    Y = O.OFDM_demodulator(x.reshape((p.Nfft + p.T_Guard, p.N_symb), order="F"), p.T_Guard)
    pc = np.asarray(p.pilotCarriers)
    q = p.pilotValues.ravel(order="F") * np.conj(Y[pc - 1, :].ravel(order="F"))
    zero = q == 0
    if not zero.any():
        return 2e-5
    pair0 = zero[1:] | zero[:-1]                                         # taus(j) reads q(j), q(j+1)
    taus = np.angle(q[1:] * np.conj(q[:-1])) / (2 * np.pi * float(pc[1] - pc[0]))
    edge = pair0[1:] != pair0[:-1]                                       # mask(j) reads taus(j - 1), taus(j)
    other = np.where(pair0[1:], taus[:-1], taus[1:])                     # the angle of that pair that is not sign-defined
    A = int(np.sum(edge & (np.abs(other) < 1e-3)))
    if A == 0:
        return 2e-5
    dif = np.abs(np.diff(taus))
    kept = taus[1:][(dif < 1e-3) & (dif != 0)][pc.size:]
    assert kept.size > 2 * A, "too few pilot-pair angles pass the mask for a tau bound: pick another stream"
    span = max(kept.max(), 0.0) - min(kept.min(), 0.0)
    return 2e-5 + 2 * A * span / (kept.size - 2 * A)


def _close(a, r, tol):      # NaN is a legitimate result of the reference algorithm (mean of an empty selection)
    return (np.isnan(a) and np.isnan(r)) or abs(a - r) < tol


def _host(ctx, out, B, p):
    h = {k: v.cpu().numpy() for k, v in out.items() if k not in ("bits", "near") and v is not None}
    h["bits"] = ctx.host_bits(out["bits"], B * p.stream_bits).reshape(B, -1)
    return h


def _check(p, out, bits, rxs, refs, flags, scramble, near_eps, tiled=1, counters=True):
    """out (host arrays of rx_chain_t4_fused, B = n * tiled streams, stream b a copy of b % n) against the oracle's refs of the
    n distinct streams.  Every stream: TgPosition, IFO and fail exact, NaN-ness of the estimates.  Streams on which the oracle
    synchronises (BER < 0.2, `Main_model_Task_4.m:367`) also: FreqOffset and tau to 2e-5, the phase inside t4_phase_bounds
    +- 2e-3, H (exp(j dphi) taken out) to 1e-3 or all-NaN with the oracle's, decisions up to _slack, symbols decided from an exact
    zero bit for bit.  Counters {errors, bits, near}."""
    td, fd, mp = flags
    n = len(refs)
    B = n * tiled
    got = out["bits"]
    full = 0
    lo_near = hi_near = 0
    all_full = True
    for b in range(n):
        ref = refs[b]
        for t in range(1, tiled):       # copies decode alike: every kernel's arithmetic is per stream
            c = b + t * n
            assert np.array_equal(got[c], got[b]), c
            for k in ("TgPosition", "IFO", "fail", "FreqOffset", "tau", "phase_shift", "H"):
                if k in out:
                    assert np.array_equal(out[k][c], out[k][b], equal_nan=True), (k, c)
        if td or fd:
            assert out["TgPosition"][b] == ref["TgPosition"] and out["fail"][b] == ref["fail"], b
            assert np.isnan(out["tau"][b]) == np.isnan(ref["tau"]) and np.isnan(out["phase_shift"][b]) == np.isnan(ref["phase_shift"]), b
        assert out["IFO"][b] == (ref["IFO"] if fd else 0), b
        ber = np.mean(ref["bits"] != bits[b])
        if ber >= 0.2:
            all_full = False
            continue
        full += 1
        dphi = dtau = 0.0
        if td or fd:
            assert _close(out["FreqOffset"][b], ref["FreqOffset"], 2e-5), b
            assert _close(out["tau"][b], ref["tau"], _tau_tol(p, rxs[b], ref, td, fd)), (b, out["tau"][b], ref["tau"])
            if not np.isnan(ref["phase_shift"]):
                lo, hi = t4_phase_bounds(p, rxs[b], ref, td, fd)
                assert lo - 2e-3 < out["phase_shift"][b] < hi + 2e-3, (b, lo, out["phase_shift"][b], hi)
                dphi = out["phase_shift"][b] - ref["phase_shift"] if fd else 0.0
                dtau = out["tau"][b] - ref["tau"] if td else 0.0
        # H carries fine_sync's correction exp(j (2 pi tau k + phase)) (`fine_sync.m:38-58`): the estimates' differences come out
        ramp = np.exp(-1j * (dphi + 2 * np.pi * dtau * np.arange(p.N_carrier)))
        if mp and "H" in out:
            Href = ref["H"][:p.N_carrier]
            if np.all(np.isfinite(Href)):
                assert rel_err(out["H"][b] * ramp, Href) < 1e-3, b
            else:
                assert np.all(np.isnan(out["H"][b].real)), b
        # decisions: raw (pre-descrambler) bits differ only inside symbols within the slack of a decision boundary
        slack = _slack(p, ref, abs(dphi) + 2 * np.pi * abs(dtau) * p.N_carrier, mp)
        raw = OC.scramble_frames(p, got[b], fast=True) if scramble else got[b]
        flipped = np.unique(np.flatnonzero(raw != ref["raw_bits"]) // p.bps)
        m = O.near_margin(ref["rx_iq"], p.Constellation)
        if flipped.size:
            assert np.all(m[flipped] < slack), (b, np.sort(m[flipped])[-3:], slack)
        zero = np.flatnonzero(ref["rx_iq"] == 0)          # data carriers past N_carrier: G = 0 on both sides
        assert not np.isin(zero, flipped).any(), b
        assert int(np.sum(got[b] != ref["bits"])) <= 3 * p.bps * flipped.size
        lo_near += int(np.sum(m < near_eps - slack))
        hi_near += int(np.sum(m < near_eps + slack))
    assert full >= 1, "no stream of this case synchronises in the oracle"
    if not counters:
        return
    counts = out["counts"]
    assert counts[1] == B * p.stream_bits
    assert counts[0] == int(np.sum(got != np.tile(bits, (tiled, 1))))
    if near_eps <= 0:
        assert counts[2] == 0
    elif all_full:
        assert tiled * lo_near <= counts[2] <= tiled * hi_near, (tiled * lo_near, int(counts[2]), tiled * hi_near)


# ------------------------------------------------------------------------------------------------------------- kernel witness
_W = Registry()
CHAIN = ("rx_t4_fast_kernel", "rx_t4_kernel", "t4_ifo_kernel", "t4_sym_kernel", "t4_post_kernel", "tx1024_kernel", "tx_chain_kernel")


def F(k2n, q16, near):
    return ("rx_t4_fast_kernel", (k2n, q16, near))


def POST(q16, near, stats=False):
    return ("t4_post_kernel", (q16, near, stats))


def SYM(k2n):
    return ("t4_sym_kernel", (k2n,))


IFOK = ("t4_ifo_kernel", ())
GEN = ("rx_t4_kernel", ())
TX1024 = ("tx1024_kernel", ())
GEN_TX = ("tx_chain_kernel", ("float",))


def split(k2n, q16, near, fd=True):
    return ([IFOK] if fd else []) + [SYM(k2n), POST(q16, near)]


def _expect(kernels, want, case):
    """The chain kernels that ran, in launch order, must be exactly `want`; records what was seen for the coverage test."""
    if not _W.record(kernels, case):
        return
    chain = [k for k in kernels if k[0] in CHAIN]
    assert chain == list(want), f"{case}: expected {want}, the profiler saw {kernels}"


def _run(ctx, lp, rx_d, bd, flags, near_eps, want, case, monkeypatch, env=None):
    if env:
        monkeypatch.setenv(env, "1")
    out, kernels = witness(lambda: ctx.rx_chain_t4_fused(lp, rx_d, tx_bits_dev=bd, time_desync=flags[0], freq_desync=flags[1],
                                                        mp_desync=flags[2], near_eps=near_eps, want_H=True))
    if env:
        monkeypatch.delenv(env)
    _expect(kernels, want, case)
    return out


# ------------------------------------------------------------------------------------------------------------- RX matrix
# id: (link parameters, options, expected chain kernels).  Options: streams (see T4_STREAMS), near (near_eps), scramble,
# flags (time/freq/mp_desync), B (streams in the call: the distinct ones tiled up to at least B), env (a switch set for the call),
# seed (of the payloads and the noise; by default one from the id).  The 52-bit frames of 16 carriers run without the
# synchroniser: three pilots leave the reference's fine_sync without a usable estimate.
RX_CASES = {
    # fused, K2N = 13: N_carrier <= 416
    "f13_q16_near_task4": (dict(S=50), dict(streams=T4_STREAMS, near=NEAR, corners=[(5, "ifo_ge1")]), [F(13, True, True)]),
    "f13_q16_nc416_unaligned": (dict(Nc=416, S=50, reg=True), dict(), [F(13, True, False)]),
    "f13_qpsk_near_reg": (dict(con="QPSK", reg=True), dict(near=NEAR), [F(13, False, True)]),
    "f13_8psk_s50": (dict(con="8PSK", S=50), dict(), [F(13, False, False)]),
    # fused, K2N = 32: N_carrier >= 417, streams short enough for 111 KB of shared memory
    "f32_q16_nc417_near": (dict(Nc=417, S=50), dict(near=NEAR, seed=5), [F(32, True, True)]),
    "f32_q16_nc800_s25": (dict(Nc=800, S=25), dict(), [F(32, True, False)]),
    "f32_bpsk_nc1024_s15_near": (dict(Nc=1024, S=15, con="BPSK", reg=True), dict(streams=FRACTIONAL, near=NEAR), [F(32, False, True)]),
    "f32_qpsk_nc800_s25": (dict(Nc=800, S=25, con="QPSK"), dict(), [F(32, False, False)]),
    "f32_8psk_nc1024_s15_near": (dict(Nc=1024, S=15, con="8PSK"), dict(streams=FRACTIONAL, near=NEAR), [F(32, False, True)]),
    # descrambler frame geometry: aligned 16QAM frames starting at every nibble of a word (the word path's history branch),
    # frames of 52 bits (< 64: frame by frame), scrambling off, data carriers past N_carrier (decided from 0)
    "f13_q16_nibbles_nc60": (dict(Nc=60, S=8, SpF=1, reg=True), dict(near=NEAR, corners=[(1, "nan_tau")]), [F(13, True, True)]),
    "f32_q16_nibbles_nc418": (dict(Nc=418, S=16, SpF=1), dict(), [F(32, True, False)]),
    "f13_q16_frame52_nc16": (dict(Nc=16, S=8, SpF=1, reg=True), dict(streams=[(0, 0.0)] * 3, flags=(0, 0, 1), near=NEAR), [F(13, True, True)]),
    "f13_q16_noscr": (dict(), dict(scramble=False, near=NEAR), [F(13, True, True)]),
    "f32_qpsk_noscr_nc600": (dict(Nc=600, con="QPSK"), dict(scramble=False), [F(32, False, False)]),
    "f13_q16_past_nc": (dict(past=4, reg=True), dict(near=NEAR), [F(13, True, True)]),
    "f32_8psk_past_nc": (dict(Nc=700, past=7, con="8PSK"), dict(), [F(32, False, False)]),
    # symbol counts: S < 7 (first round of n_first = S symbols), S = 9 (no multiple of 8)
    "f13_q16_s5": (dict(S=5), dict(near=NEAR), [F(13, True, True)]),
    "f13_q16_s9_spf3": (dict(S=9, SpF=3, reg=True), dict(), [F(13, True, False)]),
    "f32_bpsk_s1_off": (dict(Nc=500, S=1, SpF=1, con="BPSK"), dict(streams=[(0, 0.0)] * 3, flags=(0, 0, 1)), [F(32, False, False)]),
    # guards: 16 (aligned autocorrelation windows), 17 (unaligned), 1024; 0 and 1 only without the detector (W >= 16)
    "f13_q16_tg16": (dict(Tg=16), dict(near=NEAR), [F(13, True, True)]),
    "f13_qpsk_tg17": (dict(Tg=17, con="QPSK"), dict(), [F(13, False, False)]),
    "f32_q16_tg1024": (dict(Nc=500, Tg=1024), dict(near=NEAR), [F(32, True, True)]),
    "f13_q16_tg0_off": (dict(Tg=0), dict(streams=[(0, 0.0)] * 3, flags=(0, 0, 1), near=NEAR), [F(13, True, True)]),
    "f32_8psk_tg1_off": (dict(Nc=600, Tg=1, con="8PSK"), dict(streams=[(0, 0.0)] * 3, flags=(0, 0, 1)), [F(32, False, False)]),
    # estimator corners (asserted on the oracle's estimates by `corners`): IFO >= 1, NaN tau, IFO = -1 (no bin above 0.77 once
    # scaled), the detector's fallback on noise (TgPosition 65, fail = 1), and a CFO of 30.4 on a 1,000-carrier band, where
    # the wrapped top carriers reach the IFO search's first bins before the pilot does (IFO 0 in the oracle: the device must
    # agree; a stream whose IFO gather wraps and still decides those carriers needs them under 0.77 in a window that
    # straddles two symbols, which no stream makes dependable)
    # the detector's fallback on noise (TgPosition 65, fail = 1)
    "f32_q16_cfo30_nc1000": (dict(Nc=1000, S=15), dict(streams=[(1152, 30.4), (900, 0.24), (611, 3.3)], near=NEAR, corners=[(0, "ifo0"), (2, "ifo_ge1")]),
                             [F(32, True, True)]),
    "f13_q16_ifo_minus1_noise": (dict(), dict(streams=[(900, 0.24, 0.25), (611, 0.1), "noise"], near=NEAR, corners=[(0, "ifo_minus1"), (2, "fail")]),
                                 [F(13, True, True)]),
    # split chain (B >= 512): t4_sym_kernel<13 / 32>, the four t4_post_kernel<Q, NEAR, false>, 16QAM with Nd % 4 != 0 aligned
    "s13_q16_near": (dict(reg=True), dict(B=512, near=NEAR, streams=T4_STREAMS, corners=[(0, "nan_tau"), (5, "ifo_ge1")]), split(13, True, True)),
    "s13_qpsk": (dict(con="QPSK"), dict(B=512), split(13, False, False)),
    "s32_8psk_near": (dict(Nc=800, con="8PSK"), dict(B=512, near=NEAR), split(32, False, True)),
    "s32_q16_nd347_aligned": (dict(Nc=418, S=16, SpF=1), dict(B=512), split(32, True, False)),
    "s32_bpsk_ifo_minus1": (dict(Nc=600, con="BPSK"), dict(B=512, streams=[(900, 0.24, 0.15), (611, 3.3), (1, 0.49)], corners=[(0, "ifo_minus1")]),
                            split(32, False, False)),
    # fallbacks: split -> fused (Nd > S * Np; Np > 256 pilots; unaligned streams beyond one pass), -> generic (shared memory,
    # also with 342 pilots; the switch; Nfft != 1024: fine_sync's nn = 0:1023 fixes time_desync to Nfft = 1024, so those run
    # without it)
    "fb_fused_s1_nd_gt_snp": (dict(S=1, SpF=1), dict(B=512, streams=[(0, 0.0)] * 2, flags=(0, 0, 1), near=NEAR), [F(13, True, True)]),
    "fb_fused_unaligned_b16385": (dict(S=5), dict(B=16385, near=NEAR), [F(13, True, True)]),
    "fb_gen_smem_nc800_s50": (dict(Nc=800, S=50), dict(near=NEAR), [GEN]),
    "fb_fused_np342": (dict(Nc=1024, S=5, pct=30), dict(B=512, streams=FRACTIONAL, near=NEAR), [F(32, True, True)]),
    "fb_gen_smem_np342": (dict(Nc=1024, S=15, pct=30), dict(streams=FRACTIONAL), [GEN]),
    "fb_gen_no_fast": (dict(reg=True), dict(env="OFDM_B200_NO_FAST", near=NEAR), [GEN]),
    "fb_gen_nfft256": (dict(Nfft=256, Nc=200, Tg=32), dict(flags=(0, 1, 1), streams=[(0, 0.2), (0, 2.3), (0, -0.4)]), [GEN]),
    "fb_gen_nfft512": (dict(Nfft=512, Nc=400, Tg=64, con="QPSK"), dict(flags=(0, 1, 1), streams=[(0, 0.2), (0, 2.3), (0, -0.4)]), [GEN]),
    "fb_gen_nfft2048": (dict(Nfft=2048, Nc=800, Tg=256, S=5), dict(flags=(0, 1, 1), streams=[(0, 0.2), (0, 2.3), (0, -0.4)], near=NEAR), [GEN]),
}
FALLBACKS = [k for k in RX_CASES if k.startswith("fb_gen_")]


def _rx_case(G, monkeypatch, case, link, opt, want):
    p = _link(**link)
    scramble = opt.get("scramble", True)
    flags = opt.get("flags", (1, 1, 1))
    near_eps = opt.get("near", 0.0)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p, scramble)
    bits, rxs, refs = _make_streams(p, opt.get("streams", DEFAULT), opt.get("seed", sum(map(ord, case))), scramble, flags)
    n = len(refs)
    tiled = -(-opt.get("B", n) // n)
    B = n * tiled
    rx_d = ctx.cplx(np.tile(rxs, (tiled, 1)))
    bd = ctx.bits(np.tile(bits, (tiled, 1)).ravel())
    corner = {"nan_tau": lambda r: np.isnan(r["tau"]), "ifo_minus1": lambda r: r["IFO"] == -1, "ifo0": lambda r: r["IFO"] == 0,
              "ifo_ge1": lambda r: r["IFO"] >= 1, "fail": lambda r: r["fail"] == 1}
    for b, what in opt.get("corners", ()):        # the property the stream was chosen for holds in the oracle
        assert corner[what](refs[b]), (case, b, what)
    out = _run(ctx, lp, rx_d, bd, flags, near_eps, want, case, monkeypatch, opt.get("env"))
    _check(p, _host(ctx, out, B, p), bits, rxs, refs, flags, scramble, near_eps, tiled)
    return ctx, lp, p, rx_d, bd, bits, rxs, refs


@pytest.mark.parametrize("case", list(RX_CASES))
def test_rx_matrix_against_oracle(G, monkeypatch, case):
    link, opt, want = RX_CASES[case]
    _rx_case(G, monkeypatch, case, link, opt, want)
    _W.ran.add(case)


def test_rx_split_and_fused_agree_on_the_word_path(G, monkeypatch):
    """16QAM with Nd = 347 (Nd % 4 != 0) on aligned streams: the split chain's post kernel decides frame by frame while the fused
    kernel takes its word path (`chain_rx_t4.cu`, raw words of eight nibbles).  On the same 512 streams both give the same
    integer estimates and the same bits but for near-boundary symbols."""
    link, opt, want = RX_CASES["s32_q16_nd347_aligned"]
    ctx, lp, p, rx_d, bd, bits, rxs, refs = _rx_case(G, monkeypatch, "s32_q16_nd347_aligned_again", link, opt, want)
    B = rx_d.shape[0]
    s = _host(ctx, ctx.rx_chain_t4_fused(lp, rx_d, tx_bits_dev=bd, near_eps=NEAR, want_H=True), B, p)
    f = _host(ctx, _run(ctx, lp, rx_d, bd, (1, 1, 1), NEAR, [F(32, True, True)], "fused_word_path", monkeypatch, "OFDM_B200_T4_FUSED"), B, p)
    for k in ("TgPosition", "IFO", "fail"):
        assert np.array_equal(s[k], f[k]), k
    assert int(np.sum(s["bits"] != f["bits"])) <= 3 * p.bps * int(s["counts"][2] + f["counts"][2])
    assert s["counts"][1] == f["counts"][1]


def test_rx_rejects_a_stream_beyond_every_kernel(G):
    """N_carrier 400 with S = 200 needs 236.7 KB of shared memory in the generic kernel: an error with its message, no launch."""
    p = _link(S=200)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rx_d = ctx.cplx(np.zeros((2, p.stream_len), dtype=np.complex64))
    with pytest.raises(G.OfdmError, match="shared memory"):
        ctx.rx_chain_t4_fused(lp, rx_d)


def test_rx_rejects_data_past_n_carrier_without_the_equaliser(G):
    """Without estimate_channel / equalize_signal (mp_desync = 0) the reference decides a data carrier past N_carrier from its
    demodulated bin; every Task-4 kernel keeps only the N_carrier first bins, so the call refuses the layout instead of
    deciding those symbols from 0.  With the equaliser they are 0 in the reference too (f13_q16_past_nc)."""
    p = _link(past=4)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rx_d = ctx.cplx(np.zeros((2, p.stream_len), dtype=np.complex64))
    for flags in ((1, 1, 0), (0, 0, 0)):
        with pytest.raises(G.OfdmError, match="past N_carrier"):
            ctx.rx_chain_t4_fused(lp, rx_d, time_desync=flags[0], freq_desync=flags[1], mp_desync=flags[2])


# ------------------------------------------------------------------------------------------------------------- receiver stages
FLAG_SETS = [(t, f, m) for t in (0, 1) for f in (0, 1) for m in (0, 1)]


@pytest.mark.parametrize("path", ["fused", "split", "generic"])
@pytest.mark.parametrize("flags", FLAG_SETS, ids=lambda f: "td%d_fd%d_mp%d" % f)
def test_rx_receiver_stages_against_oracle(G, monkeypatch, flags, path):
    """All eight time / freq / mp_desync combinations on each path against OC.rx_chain_task4 with the same stages.  The streams
    carry only the impairments the enabled stages correct (an STO without time_desync, or a CFO without freq_desync, leaves
    the reference itself unsynchronised)."""
    td, fd, mp = flags
    spec = [(611 if td else 0, 0.24 if fd else 0.0), (1 if td else 0, 3.3 if fd else 0.0), (150 if td else 0, -0.3 if fd else 0.0)]
    p = _link(Nc=600 if path == "split" else 400, reg=True)
    k2n = 32 if p.N_carrier > 416 else 13
    want = {"fused": [F(k2n, True, True)], "split": split(k2n, True, True, fd), "generic": [GEN]}[path]
    opt = dict(streams=spec, flags=flags, near=NEAR, B=512 if path == "split" else 3, env="OFDM_B200_NO_FAST" if path == "generic" else None)
    case = "stages_%s_td%d_fd%d_mp%d" % ((path,) + flags)
    _rx_case(G, monkeypatch, case, dict(Nc=p.N_carrier, reg=True), opt, want)


# ------------------------------------------------------------------------------------------------------------- batch geometry
@pytest.fixture(scope="module")
def batch_streams(G):
    """511 distinct Task-4 streams: eight impaired oracle streams tiled, then device noise at 30 dB (a Philox stream each)."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    p = _link(S=50, reg=True)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    bits, rxs, _ = _make_streams(p, T4_STREAMS, 5, flags=(1, 1, 1))
    Bmax = 511
    reps = -(-Bmax // len(T4_STREAMS))
    rx_d = ctx.add_noise(ctx.cplx(rxs).repeat(reps, 1)[:Bmax].contiguous(), 30.0, seed=3)[0]
    bits_all = np.tile(bits, (reps, 1))[:Bmax]
    ctx.sync()
    return dict(sms=sms, p=p, lp=lp, Bmax=Bmax, rx_d=rx_d, bits=bits_all, bd=ctx.bits(bits_all.ravel()), rx=rx_d.cpu().numpy())


def test_batch_geometry_around_the_persistent_grid(G, monkeypatch, batch_streams):
    """The fused kernel at B = 1, 2 SMs - 1, 2 SMs, 2 SMs + 1 and 511 (its persistent loop and per-CTA parking area): stream b of
    every batch is bit-identical to stream b of the 511-stream call (the arithmetic is per stream), and streams 0, 510,
    grid - 1, grid and four random ones of that call match the oracle."""
    bs = batch_streams
    p, lp = bs["p"], bs["lp"]
    ctx = G.default_context("f32")
    grid = 2 * bs["sms"]
    words = p.stream_bits // 32

    def call(B):
        out = _run(ctx, lp, bs["rx_d"][:B], bs["bd"][:B * words], (1, 1, 1), NEAR, [F(13, True, True)], f"batch_{B}", monkeypatch)
        return _host(ctx, out, B, p)

    full = call(bs["Bmax"])
    for B in (1, grid - 1, grid, grid + 1):
        part = call(B)
        for k in ("bits", "TgPosition", "IFO", "fail", "FreqOffset", "tau", "phase_shift", "H"):
            assert np.array_equal(part[k], full[k][:B], equal_nan=True), (B, k)
        assert part["counts"][0] == int(np.sum(part["bits"] != bs["bits"][:B])) and part["counts"][1] == B * p.stream_bits
    rng = np.random.default_rng(grid)
    sample = sorted({0, bs["Bmax"] - 1, grid - 1, grid} | set(rng.integers(0, bs["Bmax"], 4).tolist()))
    refs = [OC.rx_chain_task4(p, bs["rx"][b].astype(np.complex128), bs["bits"][b]) for b in sample]
    for r, b in zip(refs, sample):
        r["fail"] = int(_detector_failed(bs["rx"][b].astype(np.complex128), p.T_Guard, p.Nfft))
    assert full["counts"][0] == int(np.sum(full["bits"] != bs["bits"])) and full["counts"][1] == bs["Bmax"] * p.stream_bits
    assert full["counts"][2] > 0
    sub = {k: v[sample] for k, v in full.items() if k != "counts"}
    _check(p, sub, bs["bits"][sample], [bs["rx"][b] for b in sample], refs, (1, 1, 1), True, NEAR, counters=False)


def test_split_chain_two_passes_match_single_calls(G, monkeypatch):
    """B = 16,384 + 549 aligned streams run the split chain in two passes (T4_SPLIT_CHUNK): the second pass offsets tg / fo / ifo /
    tx_bits / out_bits / H / tau / phase by the pass start.  Every stream of the second pass must be bit-identical to the same
    stream in a call of its own, and the counters the sum of the two calls'."""
    import torch
    p = _link(S=10, reg=True)                     # 13,280 bits a stream (aligned), 11,520 samples
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    bits, rxs, _ = _make_streams(p, T4_STREAMS, 11)
    CH, extra = 16384, 549                          # the second pass alone (>= 512 streams) takes the split chain too
    B = CH + extra
    reps = -(-B // len(T4_STREAMS))
    rx_d = ctx.add_noise(ctx.cplx(rxs).repeat(reps, 1)[:B].contiguous(), 30.0, seed=12)[0]
    words = p.stream_bits // 32
    bd = ctx.bits(bits.ravel()).repeat(reps)[:B * words].contiguous()
    whole = _run(ctx, lp, rx_d, bd, (1, 1, 1), NEAR, split(13, True, True) * 2, "split_two_passes", monkeypatch)
    tail = _run(ctx, lp, rx_d[CH:].contiguous(), bd[CH * words:].contiguous(), (1, 1, 1), NEAR, split(13, True, True), "split_tail", monkeypatch)
    head = _run(ctx, lp, rx_d[:CH].contiguous(), bd[:CH * words].contiguous(), (1, 1, 1), NEAR, split(13, True, True), "split_head", monkeypatch)
    assert torch.equal(whole["bits"][CH * words:], tail["bits"]) and torch.equal(whole["bits"][:CH * words], head["bits"])
    for k in ("TgPosition", "IFO", "fail", "FreqOffset", "tau", "phase_shift", "H"):
        a, t = whole[k][CH:], tail[k]
        if a.is_complex():
            a, t = torch.view_as_real(a), torch.view_as_real(t)
        assert torch.equal(torch.nan_to_num(a, nan=7.0), torch.nan_to_num(t, nan=7.0)) and torch.equal(a.isnan(), t.isnan()), k
    assert torch.equal(whole["counts"], head["counts"] + tail["counts"])
    del rx_d, whole, tail, head
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------- optional outputs
@pytest.mark.parametrize("path", ["fused", "split"])
def test_optional_outputs_and_buffer_hygiene(G, monkeypatch, path):
    """Outputs pre-filled with garbage (0xA5A5A5A5, NaN, -1) come back exactly as a call on zeroed buffers writes them; each of
    out_bits, tx_bits, counts, tg, fo, ifo, tau, phase, H and fail omitted in turn leaves the others as they were; the counters
    accumulate over calls; ifo reads 0 with freq_desync off."""
    import torch
    p = _link(Nc=418, S=16, SpF=1, reg=True)            # aligned 16QAM, Nd = 347
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    bits, rxs, _ = _make_streams(p, T4_STREAMS, 31)
    tiled = 64 if path == "split" else 1
    B = len(T4_STREAMS) * tiled
    rx_d = ctx.cplx(np.tile(rxs, (tiled, 1)))
    tx_d = ctx.bits(np.tile(bits, (tiled, 1)).ravel())
    words = (B * p.stream_bits + 31) // 32
    dev = ctx.device
    want = split(32, True, True) if path == "split" else [F(32, True, True)]
    NAMES = ("out_bits", "counts", "tg", "fo", "ifo", "tau", "phase", "H", "fail")

    def call(skip=(), counts=None, fd=1, zero=False):
        fill = (lambda shape, dt, v: torch.zeros(shape, dtype=dt, device=dev)) if zero else \
            (lambda shape, dt, v: torch.full(shape, v, dtype=dt, device=dev))
        o = dict(out_bits=fill((words,), torch.int32, -0x5A5A5A5B),       # 0xA5A5A5A5
                 counts=torch.zeros(3, dtype=torch.int64, device=dev) if counts is None else counts,
                 tg=fill((B,), torch.int32, -1), fo=fill((B,), torch.float64, np.nan), ifo=fill((B,), torch.int32, -1),
                 tau=fill((B,), torch.float64, np.nan), phase=fill((B,), torch.float64, np.nan),
                 H=fill((B, p.N_carrier), torch.complex64, complex(np.nan, np.nan)), fail=fill((B,), torch.int32, -1))
        a = {k: (None if k in skip else v) for k, v in o.items()}
        ctx._chk(ctx.lib.ofdm_rx_chain_t4_ex(ctx.h, C.byref(lp), ctx.p(rx_d), B, 1, fd, 1, ctx.p(None if "tx_bits" in skip else tx_d),
                                             ctx.p(a["out_bits"]), ctx.p(a["counts"]), ctx.p(a["tg"]), ctx.p(a["fo"]), ctx.p(a["ifo"]),
                                             ctx.p(a["tau"]), ctx.p(a["phase"]), ctx.p(a["H"]), C.c_double(NEAR), ctx.p(a["fail"])))
        ctx.sync()
        return {k: (torch.view_as_real(v) if v.is_complex() else v) for k, v in a.items() if v is not None}

    def same(x, y):
        return torch.equal(torch.nan_to_num(x, nan=7.0), torch.nan_to_num(y, nan=7.0)) and torch.equal(x.isnan(), y.isnan()) \
            if x.is_floating_point() else torch.equal(x, y)

    if path == "fused":
        monkeypatch.setenv("OFDM_B200_T4_FUSED", "1")
    ref = call(zero=True)
    assert int(ref["counts"][0]) > 0 and int(ref["counts"][2]) > 0
    got, kernels = witness(call)
    _expect(kernels, want, f"hygiene_{path}")
    for k in NAMES:
        assert same(got[k], ref[k]), k
    for skip in NAMES:
        got = call(skip=(skip,))
        for k in got:
            assert same(got[k], ref[k]), (skip, k)
    got = call(skip=("tx_bits",))
    assert int(got["counts"][0]) == 0 and int(got["counts"][1]) == B * p.stream_bits and int(got["counts"][2]) == int(ref["counts"][2])
    for k in NAMES[2:] + ("out_bits",):
        assert same(got[k], ref[k]), k
    acc = torch.zeros(3, dtype=torch.int64, device=dev)
    call(counts=acc)
    call(counts=acc)
    assert torch.equal(acc, 2 * ref["counts"])
    off, kernels = witness(lambda: call(fd=0))
    _expect(kernels, split(32, True, True, fd=False) if path == "split" else [F(32, True, True)], f"hygiene_{path}_fd0")
    assert int(off["ifo"].abs().sum()) == 0


# ------------------------------------------------------------------------------------------------------------- TX matrix
# id: (link parameters, scramble, expected kernel).  N_carrier 3 is the narrowest band that holds the two pilots the library
# requires and a data carrier.
TX_CASES = {
    "nc31_qpsk_tg0_s1": (dict(Nc=31, Tg=0, S=1, SpF=1, con="QPSK", reg=True), True, TX1024),
    "nc32_8psk_tg1": (dict(Nc=32, Tg=1, con="8PSK"), True, TX1024),
    "nc33_q16_noscr_s9": (dict(Nc=33, S=9, SpF=1), False, TX1024),
    "nc16_q16_fb52_s9": (dict(Nc=16, S=9, SpF=1, reg=True), True, TX1024),
    "nc1024_q16_tg1023": (dict(Nc=1024, Tg=1023, reg=True), True, TX1024),
    "nc1024_bpsk_tg1024_s9": (dict(Nc=1024, Tg=1024, S=9, SpF=3, con="BPSK"), True, TX1024),
    "nc400_8psk_noscr_s9": (dict(S=9, SpF=9, con="8PSK"), False, TX1024),
    "nc3_bpsk_fb1_noscr": (dict(Nc=3, pct=50, con="BPSK", S=9, SpF=1), False, TX1024),      # one data carrier: frames of 1 bit
    "nc3_bpsk_fb1": (dict(Nc=3, pct=50, con="BPSK", S=9, SpF=1, reg=True), True, TX1024),
    "fb_past_nc": (dict(past=4), True, GEN_TX),
    "fb_smem_s250": (dict(S=250), True, GEN_TX),              # frames * (fw + 1) = 50 * 209 > 5,632 words
}


@pytest.mark.parametrize("case", list(TX_CASES))
def test_tx1024_matrix_against_oracle(G, case):
    link, scramble, want = TX_CASES[case]
    p = _link(**link)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p, scramble)
    rng = np.random.default_rng(sum(map(ord, case)))
    B = 3
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    (tx, ps), kernels = witness(lambda: ctx.tx_chain(lp, ctx.bits(bits.ravel()), B, want_power=True))
    _expect(kernels, [want], f"tx_{case}")
    _W.ran.add(f"tx_{case}")
    tx_h = tx.cpu().numpy().reshape(B, -1)
    ps = ps.cpu().numpy()
    for b in range(B):
        ref, _, _ = OC.tx_chain(p, bits[b], scramble=scramble, fast=True)
        assert rel_err(tx_h[b], ref) < 2e-6, b
        assert abs(ps[b] / np.sum(np.abs(ref) ** 2) - 1) < 1e-5, b


# ------------------------------------------------------------------------------------------------------------- sweeps
def _sweep_link(Nc, frames, con, alternate=True):
    """The Task-4 layout at N_carrier Nc, 5 symbols a frame; Task 3's pilots are all +a (alternate=False)."""
    p = OC.LinkParams(Nfft=1024, N_carrier=Nc, T_Guard=128, Amount_OFDM_Frames=frames, Amount_ODFM_SpF=5, Constellation=con)
    p.pilotCarriers, p.dataCarriers = O.pilot_layout_percent(Nc, 15, 1024, last_gap=2)
    p.pilotValues, _ = OC.make_pilot_values(len(p.pilotCarriers), p.N_symb, con, 4.0 / 3.0, alternate)
    return p


def _witnessed(kernels, want, case):
    """Every kernel of `want` was launched (the sweeps launch channel and payload kernels around them)."""
    if _W.record(kernels, case):
        assert set(want) <= set(kernels), f"{case}: expected {want} among {kernels}"
    _W.ran.add(case)


@pytest.mark.parametrize("cname,snr", [("16QAM", 10.0), ("QPSK", 6.0)])
def test_sweep_sync_k32_against_oracle(G, cname, snr):
    """ofdm_sweep_sync at N_carrier 800, S = 50: the split chain's t4_sym_kernel<32> and the STATS post kernel.  The checks
    test_gpu_sweep_sync.py applies at N_carrier 400: per-stream channel error and MER, and the point's bit errors, against
    the oracle on the same streams (stages off); with every stage on, the detector's estimates and the true impairments bit
    for bit and the counters against ofdm_rx_chain_t4_ex on the same streams (that call runs its generic kernel here: the
    fused one would need 135 KB of shared memory, so its IFO and decisions agree to rounding only)."""
    from ofdm_b200 import sweep
    from test_gpu_sweep_sync import _composed, _oracle_parity
    p = _sweep_link(800, 10, cname)
    (rec, cnt, errs), kernels = witness(lambda: _oracle_parity(p, snr, 4, 8))
    _witnessed(kernels, [SYM(32), POST(cname == "16QAM", False, True)], f"sweep_sync_{cname}")
    assert np.all(np.isfinite(rec[0, 5]))
    ctx = G.default_context("f32")
    lp = ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                         p.pilotCarriers, p.pilotValues)
    n, seed = 64, 11
    rec, cnt = sweep.sync_sweep_local(ctx, lp, [30.0], n, TAPS4, seed=seed, tile=n)
    ctx.sync()
    rec, cnt = rec.cpu().numpy(), cnt.cpu().numpy()
    exp, ecnt, _, _ = _composed(ctx, lp, p, 30.0, 0, n, seed, TAPS4, None, None, (1, 1, 1))
    for f in (0, 1, 7, 8):
        assert np.array_equal(rec[0, f], exp[f]), f
    assert cnt[0, 1] == ecnt[1] and cnt[0, 2] == ecnt[2]


@pytest.mark.parametrize("cname", ["BPSK", "QPSK", "8PSK", "16QAM"])
def test_sweep_mer_k32_noise_free_against_oracle(G, cname):
    """ofdm_sweep_mer at N_carrier 800 (rx_t3_kernel<32, *>), noise-free, under the fixed STO / CFO and multipath it does not
    correct, against the oracle's Task-3 receiver: bit errors up to near-boundary symbols, MER to 1e-3 dB; without any
    impairment, no error."""
    from ofdm_b200 import sweep
    from test_gpu_sweep_mer import _oracle_stream, _s_bits
    ctx = G.default_context("f32")
    p = _sweep_link(800, 10, cname, alternate=False)
    lp = ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                         p.pilotCarriers, p.pilotValues)
    n, seed, eps = 3, 4, 1e-3
    s = _s_bits(ctx, p, n, seed, 0)
    for i, (sto, cfo, taps) in enumerate([(5, 0.0, []), (0, 0.3, []), (0, 0.0, TAPS4), (5, 0.3, TAPS4)]):
        res, kernels = witness(lambda: sweep.mer_sweep(ctx, lp, cname, [np.inf], n, taps, seed=seed, sto=sto, cfo=cfo, near_eps=eps))
        _witnessed(kernels, [("rx_t3_kernel", (32, cname == "16QAM"))], f"sweep_mer_{cname}_{i}")
        errs, mers = zip(*(_oracle_stream(p, s[j], sto, cfo, taps or None) for j in range(n)))
        got = res["counts"][0]
        assert abs(int(got[0]) - sum(errs)) <= 3 * p.bps * int(got[2]), (cname, sto, got, errs)
        assert np.max(np.abs(res["per_stream_db"][0] - np.array(mers))) < 1e-3, (cname, sto, res["per_stream_db"][0], mers)
    clean = sweep.mer_sweep(ctx, lp, cname, [np.inf], 8, seed=seed)      # no impairment: no error, MER limited by rounding only
    assert clean["counts"][0, 0] == 0 and np.all(clean["per_stream_db"] > 100.0)


@pytest.mark.parametrize("Nc,frames", [(800, 5), (400, 10)])
def test_sweep_mer_equals_the_split_chain(G, Nc, frames):
    """ofdm_sweep_mer's bins and decisions are those of ofdm_rx_chain_t4_ex(..., 0, 0, 0, ...)'s split chain on the same 512
    streams (rx_t3_kernel<32 / 13, *> against t4_sym_kernel + t4_post_kernel): the same bit errors.  At N_carrier 800 the
    streams have 5 frames: with 10 the fused kernel does not fit and ofdm_rx_chain_t4_ex runs its generic kernel instead."""
    from ofdm_b200 import sweep
    from test_gpu_sweep_sync import _composed
    ctx = G.default_context("f32")
    k2n = 32 if Nc > 416 else 13
    n, seed = 512, 9
    for cname, snr, sto, cfo, taps in (("8PSK", 9.0, 3, 0.05, TAPS4), ("16QAM", 14.0, 0, 0.0, [])):
        p = _sweep_link(Nc, frames, cname, alternate=False)
        lp = ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                             p.pilotCarriers, p.pilotValues)
        res, k1 = witness(lambda: sweep.mer_sweep(ctx, lp, cname, [snr], n, taps, seed=seed, sto=sto, cfo=cfo, tile=200))
        _witnessed(k1, [("rx_t3_kernel", (k2n, cname == "16QAM"))], f"sweep_mer_split_{Nc}_{cname}")
        (_, cnt, _, _), k2 = witness(lambda: _composed(ctx, lp, p, snr, 0, n, seed, taps, sto, cfo, (0, 0, 0)))
        _witnessed(k2, [SYM(k2n), POST(cname == "16QAM", False)], f"sweep_mer_split_ref_{Nc}_{cname}")
        assert np.array_equal(res["counts"][0, :2], cnt[:2]) and cnt[0] > 0


def test_sweep_mer_rejects_data_past_n_carrier(G):
    """Task 3 decides a data carrier past N_carrier from its (unequalised) bin, which rx_t3_kernel does not keep: refused."""
    from ofdm_b200 import sweep
    ctx = G.default_context("f32")
    p = _link(past=4)
    lp = _lp(ctx, p)
    with pytest.raises(G.OfdmError, match="past N_carrier"):
        sweep.mer_sweep(ctx, lp, "16QAM", [10.0], 4)


# ------------------------------------------------------------------------------------------------------------- coverage
def test_witness_covered_every_instantiation():
    """The cases above together launched all eight rx_t4_fast_kernel instantiations, both t4_sym_kernel, the four t4_post_kernel
    of the BER chain and the two STATS ones of ofdm_sweep_sync, the four rx_t3_kernel of ofdm_sweep_mer, t4_ifo_kernel,
    tx1024_kernel and its generic fallback, and rx_t4_kernel for every fallback reason."""
    if _W.available is False:
        pytest.skip("the profiler recorded no CUDA activity (no CUPTI): kernel identities are not observable here")
    sweeps = {f"sweep_sync_{c}" for c in ("16QAM", "QPSK")} | {f"sweep_mer_{c}_0" for c in ("BPSK", "QPSK", "8PSK", "16QAM")}
    sweeps |= {f"sweep_mer_split_{nc}_{c}" for nc in (400, 800) for c in ("8PSK", "16QAM")}
    if _W.available is None or (set(RX_CASES) | {f"tx_{c}" for c in TX_CASES} | sweeps) - _W.ran:
        pytest.skip("kernel coverage needs every RX, TX and sweep case of this module in the same session")
    want = {F(k, q, n) for k in (13, 32) for q in (False, True) for n in (False, True)}
    want |= {SYM(13), SYM(32), IFOK, TX1024, GEN_TX} | {POST(q, n) for q in (False, True) for n in (False, True)}
    want |= {POST(q, False, True) for q in (False, True)} | {("rx_t3_kernel", (k, q)) for k in (13, 32) for q in (False, True)}
    seen = set(_W.seen)
    print("Nfft-1024 kernel instantiations observed:", sorted(k for k in seen if k[0] in CHAIN + ("rx_t3_kernel",)))
    print("generic receiver observed for:", sorted(_W.seen.get(GEN, ())))
    assert len(want) == 23 and want <= seen, sorted(want - seen)
    assert set(FALLBACKS) <= _W.seen.get(GEN, set())
