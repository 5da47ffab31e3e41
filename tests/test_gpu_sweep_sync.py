"""ofdm_sweep_sync (Task 4's synchroniser and channel-estimate study over SNR) on the GPU: its records are those of the same
streams pushed through the exported calls one by one, its counters those of ofdm_sweep_ber's Task-4 chain, independent of
tile size and rank count, its MER that of the oracle's MER_func, the pins P5 / P6 of tests/test_sync_pins.py hold on the
GPU path, NaN cells are counted, every bad argument is refused with its own text, and the MEX gateway gives the same."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O
from oracle import chains as OC
from test_sync_pins import P5_RTOL, P5_SNR, P6_CFO_BOUND, P6_FAIL_AT_0DB

pytestmark = pytest.mark.gpu

TAPS4 = [[0, 1], [4, .6], [10, .3]]            # `Task 4/Main_model_Task_4.m:252-264`


def _ctx(prec="f32"):
    import ofdm_b200 as G
    return G.default_context(prec)


def _lp(ctx, p):
    return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                           p.pilotCarriers, p.pilotValues)


def _h_true(taps, Nfft, Nc):
    if not taps:
        return np.ones(Nc, dtype=np.complex128)
    h, _ = O.get_MP_channel_resp(taps, Nfft)
    k = np.arange(Nc)
    return np.array([np.sum([h[d] * np.exp(-2j * np.pi * ((d * kk) % Nfft) / Nfft) for d in np.nonzero(h)[0]]) for kk in k])


def _composed(ctx, lp, p, snr, g0, n, seed, taps, sto, cfo, flags):
    """The streams g0 .. g0 + n - 1 of the sweep rebuilt through the exported calls, received by ofdm_rx_chain_t4_ex (n >= 512:
    its split chain).  Returns (expected record [9, n], counters [4], the received streams, the payload bits)."""
    words = -(-p.stream_bits // 32)
    raw = torch.zeros(n * words, dtype=torch.int32, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(raw), n, words, seed, g0))
    s_bits = np.unpackbits(raw.cpu().numpy().view(np.uint8), bitorder="little").reshape(n, -1)[:, :p.stream_bits]
    sbits = ctx.bits(s_bits.ravel())                            # scrambled frames s; the payload is p = DeScrambler(s)
    bits = ctx.scramble(sbits, n * p.Amount_OFDM_Frames, p.frame_bits, descramble=True)
    if sto is None:
        sto_d = torch.zeros(n, dtype=torch.int32, device=ctx.device)
        cfo_d = torch.zeros(n, dtype=torch.float64, device=ctx.device)
        ctx._chk(ctx.lib.ofdm_draw_sto_cfo(ctx.h, n, seed, g0, p.Nfft + p.T_Guard, 30, ctx.p(sto_d), ctx.p(cfo_d)))
    else:
        sto_d = torch.full((n,), sto, dtype=torch.int32, device=ctx.device)
        cfo_d = torch.full((n,), cfo, dtype=torch.float64, device=ctx.device)
    lp_tx = ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers, p.pilotCarriers,
                            p.pilotValues, scramble=False)
    tx, psum = ctx.tx_chain(lp_tx, sbits, n, want_power=True)   # as ofdm_sweep_ber: the transmitter maps s itself
    h = O.get_MP_channel_resp(taps, p.Nfft)[0] if taps else np.ones(1)
    rx = ctx.channel_t4(tx.reshape(n, -1), float(snr), sto_d, cfo_d, p.Nfft, ctx.cplx(h.astype(np.complex128)), seed=seed, first_stream_id=g0,
                        power_sum=psum)
    t, f, m = flags
    out = ctx.rx_chain_t4_fused(lp, rx.reshape(n, p.N_symb, -1), tx_bits_dev=bits, time_desync=t, freq_desync=f, mp_desync=m, want_bits=False,
                                want_H=m)
    ctx.sync()
    exp = np.zeros((9, n))
    exp[0] = out["TgPosition"].cpu().numpy() if t else 0
    exp[1] = out["FreqOffset"].cpu().numpy() if f else 0
    exp[2] = out["IFO"].cpu().numpy()
    exp[3] = out["tau"].cpu().numpy()
    exp[4] = out["phase_shift"].cpu().numpy()
    if m:
        c64 = _ctx("f64")                                      # ofdm_mse on the FP32 estimate against the double true response
        Hd = torch.from_numpy(out["H"].cpu().numpy().astype(np.complex128)).to(c64.device)
        Ht = torch.from_numpy(np.tile(_h_true(taps, p.Nfft, p.N_carrier), (n, 1))).to(c64.device)
        exp[5] = c64.mse(Ht, Hd, p.N_carrier).cpu().numpy()
    else:
        exp[5] = np.nan
    exp[7] = sto_d.cpu().numpy()
    exp[8] = cfo_d.cpu().numpy()
    cnt = out["counts"].cpu().numpy()
    fail = int(out["fail"].sum()) if (t or f) else 0
    return exp, np.array([cnt[0], cnt[1], fail, int((out["IFO"] == -1).sum()) if f else 0]), rx, bits


CASES = {   # name: (params, taps, sto, cfo, (time, freq, mp), snr)
    "drawn_mp": (lambda: OC.params_task4(), TAPS4, None, None, (1, 1, 1), 30.0),
    "fixed_awgn": (lambda: OC.params_task4(), [], 150, 0.24, (1, 1, 0), 8.0),
    "clean_mp": (lambda: OC.params_task4(), TAPS4, 0, 0.0, (0, 0, 1), 10.0),
    "freq_only": (lambda: OC.params_task4(), TAPS4, 0, 2.3, (0, 1, 1), 20.0),
}


@pytest.mark.parametrize("name", list(CASES))
def test_records_equal_composed_calls(name):
    from ofdm_b200 import sweep
    mk, taps, sto, cfo, flags, snr = CASES[name]
    p = mk()
    ctx = _ctx()
    lp = _lp(ctx, p)
    spp, seed = 600, 11
    kw = dict(sto=sto, cfo=cfo) if sto is not None else {}
    rec, cnt = sweep.sync_sweep_local(ctx, lp, [snr - 6.0, snr], spp, taps, seed=seed, tile=600, time_desync=flags[0], freq_desync=flags[1],
                                      mp_desync=flags[2], **kw)
    ctx.sync()
    rec, cnt = rec.cpu().numpy(), cnt.cpu().numpy()
    exp, ecnt, _, _ = _composed(ctx, lp, p, snr, spp, spp, seed, taps, sto, cfo, flags)
    for f in (0, 1, 2, 3, 4, 7, 8):                            # the estimates and true impairments: bit for bit
        assert np.array_equal(rec[1, f], exp[f], equal_nan=True), sweep.SYNC_FIELDS[f]
    if flags[2]:
        ok = ~np.isnan(exp[5])
        assert np.array_equal(np.isnan(rec[1, 5]), ~ok)
        assert np.allclose(rec[1, 5][ok], exp[5][ok], rtol=1e-12, atol=0)
    else:
        assert np.all(np.isnan(rec[1, 5]))
    assert np.array_equal(cnt[1], ecnt)


def test_pilot_step4_layout_against_generic_kernel():
    """At 25 % pilots (101 pilots, unaligned 59,800-bit streams) ofdm_rx_chain_t4_ex runs its generic block-FFT kernel (the
    fused fast kernel would need 121 KB of shared memory), whose FP32 arithmetic differs from the split chain's in rounding
    only: the same streams give the same channel error to FP32 accuracy and the same bit errors up to a few decisions."""
    from ofdm_b200 import sweep
    p = OC.params_task4(percent=25)
    ctx = _ctx()
    lp = _lp(ctx, p)
    spp, seed, snr = 600, 11, 10.0
    rec, cnt = sweep.sync_sweep_local(ctx, lp, [snr], spp, TAPS4, seed=seed, sto=0, cfo=0.0, time_desync=False, freq_desync=False)
    ctx.sync()
    exp, ecnt, _, _ = _composed(ctx, lp, p, snr, 0, spp, seed, TAPS4, 0, 0.0, (0, 0, 1))
    rec, cnt = rec.cpu().numpy(), cnt.cpu().numpy()
    assert np.allclose(rec[0, 5], exp[5], rtol=1e-4, atol=0)
    assert cnt[0, 1] == ecnt[1] and abs(int(cnt[0, 0]) - int(ecnt[0])) <= 1e-5 * ecnt[1]


def test_counters_equal_sweep_ber():
    from ofdm_b200 import sweep
    p = OC.params_task4()
    ctx = _ctx()
    lp = _lp(ctx, p)
    snrs, spp, seed = [10.0, 25.0], 1024, 4
    ber = sweep.ber_sweep(ctx, lp, snrs, spp, TAPS4, "task4", seed=seed, tile=512)
    res = sweep.sync_sweep(ctx, lp, snrs, spp, TAPS4, seed=seed, tile=512)
    assert np.array_equal(res["counts"][:, :2], ber[:, :2]) and np.array_equal(res["counts"][:, 2], ber[:, 3])


def test_split_invariance():
    from ofdm_b200 import sweep
    p = OC.params_task4()
    ctx = _ctx()
    lp = _lp(ctx, p)
    snrs, spp, seed = [0.0, 12.0], 1100, 7
    base = sweep.sync_sweep_local(ctx, lp, snrs, spp, TAPS4, seed=seed)
    ctx.sync()
    for tile in (512, 777):
        r, c = sweep.sync_sweep_local(ctx, lp, snrs, spp, TAPS4, seed=seed, tile=tile)
        ctx.sync()
        assert torch.equal(r.nan_to_num(7.0), base[0].nan_to_num(7.0)) and torch.equal(c, base[1])
    rec = torch.zeros_like(base[0])
    cnt = torch.zeros_like(base[1])
    for rank in range(3):                                      # three ranks' calls fill one buffer
        sweep.sync_sweep_local(ctx, lp, snrs, spp, TAPS4, seed=seed, rank=rank, world=3, tile=500, rec=rec, counts=cnt)
    ctx.sync()
    assert torch.equal(rec.nan_to_num(7.0), base[0].nan_to_num(7.0)) and torch.equal(cnt, base[1])
    assert int(torch.isnan(base[0][0, 5]).sum()) > 0            # 0 dB: failed synchronisations leave NaN estimates


def test_mer_against_oracle_and_awgn_budget():
    from ofdm_b200 import sweep
    p = OC.params_task4()
    ctx = _ctx()
    lp = _lp(ctx, p)
    # per-stream MER_func of the oracle's receiver on the very streams the sweep built
    spp, seed, snr = 512, 3, 20.0
    rec, _ = sweep.sync_sweep_local(ctx, lp, [snr], spp, TAPS4, seed=seed, sto=0, cfo=0.0, time_desync=0, freq_desync=0)
    ctx.sync()
    _, _, rx, bits = _composed(ctx, lp, p, snr, 0, spp, seed, TAPS4, 0, 0.0, (0, 0, 1))
    rx_h = rx.cpu().numpy().astype(np.complex128)
    bits_h = ctx.host_bits(bits, spp * p.stream_bits).reshape(spp, -1)
    for b in range(4):
        ref = OC.rx_chain_task4(p, rx_h[b], bits_h[b], time_desync=False, freq_desync=False)
        assert abs(rec[0, 6, b].item() - O.MER_func(ref["rx_iq"], p.Constellation)) < 2e-3
    # AWGN, no impairments: mean MER = SNR + 10 log10(Nfft / (Nd + Np a^2 / E|d|^2)), the relation behind P2
    res = sweep.sync_sweep(ctx, lp, [25.0], 2048, None, seed=5, sto=0, cfo=0.0, time_desync=False, freq_desync=False)
    d, _ = O.constellation_func(p.Constellation)
    a2 = np.abs(p.pilotValues[0, 0]) ** 2 / np.mean(np.abs(d) ** 2)
    expect = 25.0 + 10 * np.log10(p.Nfft / (len(p.dataCarriers) + len(p.pilotCarriers) * a2))
    assert abs(res["mer_db"][0] - expect) < 0.1, (res["mer_db"][0], expect)


NEAR_EPS = 1e-3      # squared-distance margin under which an FP32 decision may legitimately differ from the float64 one


def _oracle_parity(p, snr, n, seed):
    """The sweep's records and counters for n streams (one point, fixed STO 0 / CFO 0, no sync stages, 3-tap channel) against
    the oracle's receiver (OC.rx_chain_task4) on the very same streams.  Per stream: the H error (field 5) to P5_RTOL, the MER
    (field 6) to 2e-3 dB; the point's bit errors exactly, up to 3 bps output bits (one raw bit feeds three descrambled ones)
    per symbol the oracle decides within NEAR_EPS of a boundary."""
    from ofdm_b200 import sweep
    ctx = _ctx()
    lp = _lp(ctx, p)
    rec, cnt = sweep.sync_sweep_local(ctx, lp, [snr], n, TAPS4, seed=seed, sto=0, cfo=0.0, time_desync=False, freq_desync=False)
    ctx.sync()
    rec, cnt = rec.cpu().numpy(), cnt.cpu().numpy()
    _, _, rx, bits = _composed(ctx, lp, p, snr, 0, n, seed, TAPS4, 0, 0.0, (0, 0, 1))
    rx_h = rx.cpu().numpy().astype(np.complex128).reshape(n, -1)
    bits_h = ctx.host_bits(bits, n * p.stream_bits).reshape(n, -1)
    H_true = np.fft.fft(O.get_MP_channel_resp(TAPS4, p.Nfft)[0], p.Nfft)[:p.N_carrier]
    d, _ = O.constellation_func(p.Constellation)
    errs = near = 0
    for b in range(n):
        ref = OC.rx_chain_task4(p, rx_h[b], bits_h[b], time_desync=False, freq_desync=False)
        e = np.mean(np.abs(ref["H"][:p.N_carrier] - H_true) ** 2)
        assert abs(rec[0, 5, b] - e) <= P5_RTOL * e, (snr, b, rec[0, 5, b], e)
        assert abs(rec[0, 6, b] - O.MER_func(ref["rx_iq"], p.Constellation)) < 2e-3
        dist = np.sort(np.abs(ref["rx_iq"][None, :] - d[:, None]) ** 2, axis=0)
        near += int(np.sum(dist[1] - dist[0] < NEAR_EPS))
        errs += ref["errors"]
    assert cnt[0, 1] == n * p.stream_bits and cnt[0, 2] == 0 and cnt[0, 3] == 0
    assert abs(int(cnt[0, 0]) - errs) <= 3 * p.bps * near, (int(cnt[0, 0]), errs, near)
    return rec, cnt, errs


@pytest.mark.parametrize("snr", P5_SNR)
def test_p5_h_error_matches_oracle(snr):
    """P5 (DESIGN §2): at the figure's layout -- 25 % pilots, step 4, unaligned 59,800-bit streams, so also the packing of the
    payload, the 5,980-bit frames of the descrambler and the generic 16QAM decision branch -- the per-stream channel error
    equals the oracle's on the same streams to FP32 accuracy, and so do the MER and the bit errors."""
    p = OC.params_task4(percent=25)
    assert len(p.pilotCarriers) == 101 and p.stream_bits % 32 != 0
    rec, _, _ = _oracle_parity(p, snr, 4, 8)
    assert np.all(np.isfinite(rec[0, 5]))


def test_qpsk_decisions_and_mer_match_oracle():
    """The nearest_idx decision branch (constellations other than 16QAM; QPSK streams of 33,200 bits are unaligned too)."""
    p = OC.params_task4(Constellation="QPSK")
    _, _, errs = _oracle_parity(p, 6.0, 4, 21)
    assert errs > 0                                            # the comparison covers decision errors, not only clean streams


def test_p6_on_gpu():
    from ofdm_b200 import sweep
    ctx = _ctx()
    p = OC.params_task4()
    lp = _lp(ctx, p)
    res = sweep.sync_sweep(ctx, lp, [0.0, 10.0, 15.0, 20.0], 2048, None, seed=9, sto=150, cfo=0.24, mp_desync=False)
    assert res["fail_rate"][0] >= P6_FAIL_AT_0DB
    fo = res["rec"][:, 1, :]
    assert np.all(res["fail_rate"][1:] == 0)
    assert np.all(np.mean(np.abs(fo[1:] - 0.24) < P6_CFO_BOUND, axis=1) >= 0.99)


def test_nan_cells_are_counted():
    from ofdm_b200 import sweep
    p = OC.params_task4()
    ctx = _ctx()
    lp = _lp(ctx, p)
    res = sweep.sync_sweep(ctx, lp, [0.0], 600, TAPS4, seed=2, sto=150, cfo=0.24)
    nan = np.isnan(res["rec"][0, 5])
    assert nan.sum() > 0 and res["h_err_nan"][0] == nan.sum()
    assert np.isfinite(res["h_err_mean"][0]) or nan.all()


def test_rejections():
    from ofdm_b200 import _cabi
    ctx = _ctx()
    p = OC.params_task4()
    lp = _lp(ctx, p)
    snr = np.array([10.0])
    rec = torch.zeros((1, 9, 4), dtype=torch.float64, device=ctx.device)
    cnt = torch.zeros((1, 4), dtype=torch.int64, device=ctx.device)

    def params(**kw):
        sp = _cabi.SyncParams()
        sp.n_snr, sp.snr_db_host, sp.streams_per_point, sp.rank, sp.world, sp.seed = 1, snr.ctypes.data_as(_cabi.pdbl), 4, 0, 1, 1
        sp.sto_max, sp.cfo_int_max, sp.time_desync, sp.freq_desync, sp.mp_desync = 1152, 30, 1, 1, 1
        for k, v in kw.items():
            setattr(sp, k, v)
        return sp

    def call(c=ctx, l=lp, s=None, r=rec, n=cnt):
        s = params() if s is None else s
        rc = c.lib.ofdm_sweep_sync(c.h, C.byref(l) if l is not None else None, C.byref(s) if s is not False else None, c.p(r), c.p(n))
        return rc, c.lib.ofdm_last_error(c.h).decode()

    assert call()[0] == 0
    ctx.sync()
    texts = set()
    bad_taps = np.array([[2000.0, 1.0]])
    for rc_want, args in [(-1, dict(l=None)), (-1, dict(s=False)), (-1, dict(r=None)), (-1, dict(n=None)),
                          (-1, dict(s=params(n_snr=0))), (-1, dict(s=params(streams_per_point=0))), (-1, dict(s=params(tile_streams=-1))),
                          (-1, dict(s=params(rank=1))), (-1, dict(s=params(sto_mode=2))), (-1, dict(s=params(sto_max=-1))),
                          (-1, dict(s=params(sto_mode=1, sto_fixed=-3))), (-1, dict(s=params(n_taps=1))),
                          (-1, dict(s=params(n_taps=1, taps_host=bad_taps.ctypes.data_as(_cabi.pdbl))))]:
        rc, text = call(**args)
        assert rc == rc_want, (args, rc, text)
        texts.add(text)
    assert len(texts) == 13                                     # every check has its own text
    c64 = _ctx("f64")
    rc, text = call(c=c64, l=_lp(c64, p))
    assert rc == -4 and "FP32" in text
    p2 = OC.params_task5(comb=4)
    rc, text = call(l=ctx.link_params(p2.Nfft, p2.T_Guard, p2.N_carrier, p2.N_symb, p2.Amount_ODFM_SpF, p2.Constellation, p2.dataCarriers,
                                      p2.pilotCarriers, p2.pilotValues))
    assert rc == -4 and "Nfft = 1024" in text


def test_mex_gateway_equals_python():
    import os
    import subprocess
    from ofdm_b200 import sweep
    from test_gpu_mex import Mex
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["make", "-C", os.path.join(root, "mex")], check=True, capture_output=True)
    mex = Mex("interleaved")
    ctx = _ctx()
    p = OC.params_task4()
    lp = _lp(ctx, p)
    reg = O.DEFAULT_REGISTER.astype(float)
    try:
        snrs, spp = [5.0, 15.0], 520
        args = [float(p.Nfft), float(p.T_Guard), float(p.N_carrier), float(p.N_symb), float(p.Amount_ODFM_SpF), p.Constellation,
                p.dataCarriers.astype(float), p.pilotCarriers.astype(float), p.pilotValues, reg]
        for sto, cfo, flags in ((-1.0, 0.0, [1.0, 1.0, 1.0]), (150.0, 0.24, [1.0, 1.0, 0.0])):
            got_r, got_c = mex.call("sweep_sync", *args, np.asarray(snrs), float(spp), np.asarray(TAPS4, dtype=float), 3.0, sto, cfo,
                                    np.asarray(flags), nout=2)
            kw = dict(sto=int(sto), cfo=cfo) if sto >= 0 else {}
            res = sweep.sync_sweep(ctx, lp, snrs, spp, TAPS4, seed=3, time_desync=bool(flags[0]), freq_desync=bool(flags[1]),
                                   mp_desync=bool(flags[2]), **kw)
            assert got_r.shape == (spp, 9 * len(snrs))
            ref = res["rec"]
            got = got_r.reshape(spp, 9, len(snrs), order="F").transpose(2, 1, 0)
            assert np.array_equal(np.nan_to_num(got, nan=7.0), np.nan_to_num(ref, nan=7.0))
            assert np.array_equal(got_c.astype(np.int64), res["counts"])
    finally:
        mex.lib.ofdm_mex_shim_exit()
