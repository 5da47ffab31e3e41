"""ofdm_sweep_mer (Task 3's BER and MER study over constellations and SNR) on the GPU: its counters and MER are those of
ofdm_sweep_sync with every receiver stage off on the same streams, and of the same streams pushed through the exported calls
one by one; noise-free it agrees with the float64 oracle under uncorrected STO, CFO and multipath; it does not depend on the
rank count or the tile size; the Task-3 pins P1 / P2 hold on it; a device group and the MEX gateway give the same; and bad
arguments are refused."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import oracle as O
import reference_pins as RP
from oracle import chains as OC

pytestmark = pytest.mark.gpu

TAPS4 = [[0, 1], [4, .6], [10, .3]]            # `Task 4/Main_model_Task_4.m:252-264`
NAMES = ("BPSK", "QPSK", "8PSK", "16QAM")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ctx(prec="f32"):
    import ofdm_b200 as G
    return G.default_context(prec)


def _lp(ctx, p):
    return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                           p.pilotCarriers, p.pilotValues)


def _sweep():
    from ofdm_b200 import sweep
    return sweep


def _s_bits(ctx, p, n, seed, g0):
    """The scrambled frames s of streams g0 .. g0 + n - 1 as the sweep draws them: (n, stream_bits) uint8."""
    words = -(-p.stream_bits // 32)
    raw = torch.zeros(n * words, dtype=torch.int32, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(raw), n, words, seed, g0))
    return np.unpackbits(raw.cpu().numpy().view(np.uint8), bitorder="little").reshape(n, -1)[:, :p.stream_bits]


@pytest.mark.parametrize("cname", NAMES)
def test_equals_sync_sweep_with_receiver_stages_off(cname):
    sweep = _sweep()
    ctx = _ctx()
    p = OC.params_task4(alternate=False, Constellation=cname)
    lp = _lp(ctx, p)
    snrs, spp = [0.0, 6.0, 12.0], 96
    res = sweep.mer_sweep(ctx, lp, cname, snrs, spp, seed=5, sto=0, cfo=0.0)
    ref = sweep.sync_sweep(ctx, lp, snrs, spp, seed=5, sto=0, cfo=0.0, time_desync=False, freq_desync=False, mp_desync=False)
    assert np.array_equal(res["counts"][:, :2], ref["counts"][:, :2])
    assert np.all(res["counts"][:, 1] == spp * p.stream_bits) and res["counts"][0, 0] > 0
    assert np.max(np.abs(res["per_stream_db"] - ref["rec"][:, 6, :])) < 1e-9


def test_equals_composed_exported_calls():
    """Streams rebuilt through ofdm_payload_bits -> pack -> ofdm_tx_chain_p -> ofdm_channel_t4_p -> ofdm_rx_chain_t4_ex(0, 0, 0)
    on the real DeScrambler(s) (512 streams: the split chain), and MER through ofdm_demodulate / ofdm_get_payload / ofdm_mer."""
    from test_gpu_sweep_sync import _composed
    sweep = _sweep()
    ctx = _ctx()
    n, seed = 512, 9
    for cname, snr, sto, cfo, taps in (("8PSK", 9.0, 3, 0.05, TAPS4), ("16QAM", 14.0, 0, 0.0, [])):
        p = OC.params_task4(alternate=False, Constellation=cname)
        lp = _lp(ctx, p)
        res = sweep.mer_sweep(ctx, lp, cname, [snr], n, taps, seed=seed, sto=sto, cfo=cfo, tile=200)
        _, cnt, rx, _ = _composed(ctx, lp, p, snr, 0, n, seed, taps, sto, cfo, (0, 0, 0))
        assert np.array_equal(res["counts"][0, :2], cnt[:2]) and cnt[0] > 0
        grid = ctx.demodulate(rx.reshape(n, p.N_symb, -1), p.Nfft, p.T_Guard)
        iq = ctx.get_payload(grid, p.dataCarriers)
        for b in range(0, n, 37):
            s = ctx.mer(iq[b].reshape(-1), cname).cpu().numpy()
            assert np.allclose(res["mer"][0, :, b], s, rtol=1e-6, atol=0), (cname, b)


def _oracle_stream(p, s, sto, cfo, taps):
    tx, _, _ = OC.tx_chain(p, s, scramble=False)
    rx = OC.impair_task4(p, tx, None, sto, cfo, taps)
    Y = O.OFDM_demodulator(rx[:p.stream_len].reshape((p.Nfft + p.T_Guard, p.N_symb), order="F"), p.T_Guard)
    iq = O.get_payload(Y, p.dataCarriers).ravel(order="F")
    d = O.demapping(-1, iq, p.Constellation)
    err = int(np.sum(OC.scramble_frames(p, d, descramble=True) != OC.scramble_frames(p, s, descramble=True)))
    _, s1, s2 = O.MER_func(iq, p.Constellation, return_sums=True)
    return err, 10 * np.log10(s1 / s2)


@pytest.mark.parametrize("cname", NAMES)
def test_noise_free_impairments_against_oracle(cname):
    sweep = _sweep()
    ctx = _ctx()
    p = OC.params_task4(alternate=False, Constellation=cname)
    lp = _lp(ctx, p)
    cases = [(5, 0.0, []), (0, 0.3, []), (0, 0.0, TAPS4), (5, 0.3, TAPS4)]
    n, seed, eps = 3, 4, 1e-3
    s = _s_bits(ctx, p, n, seed, 0)
    for sto, cfo, taps in cases:
        res = sweep.mer_sweep(ctx, lp, cname, [np.inf], n, taps, seed=seed, sto=sto, cfo=cfo, near_eps=eps)
        errs, mers = zip(*(_oracle_stream(p, s[j], sto, cfo, taps or None) for j in range(n)))
        got = res["counts"][0]
        assert abs(int(got[0]) - sum(errs)) <= 3 * p.bps * int(got[2]), (cname, sto, cfo, taps, got, errs)
        assert np.max(np.abs(res["per_stream_db"][0] - np.array(mers))) < 1e-3, (cname, sto, cfo, taps, res["per_stream_db"][0], mers)
    clean = sweep.mer_sweep(ctx, lp, cname, [np.inf], 8, seed=seed)
    assert clean["counts"][0, 0] == 0 and np.all(clean["per_stream_db"] > 100.0)


def test_independent_of_rank_count_and_tile():
    sweep = _sweep()
    ctx = _ctx()
    p = OC.params_task4(alternate=False)
    lp = _lp(ctx, p)
    cons = ["BPSK", "QPSK", "8PSK", "16QAM", "QPSK"]
    snrs, spp = [4.0, 8.0, 10.0, 16.0, 6.0], 50
    kw = dict(seed=13, sto=[0, 2, 0, 1, 3], cfo=[0.0, 0.02, 0.05, 0.0, 0.01], near_eps=1e-2)
    ref_m, ref_c = sweep.mer_sweep_local(ctx, lp, cons, snrs, spp, TAPS4, **kw)
    ctx.sync()
    ref_m, ref_c = ref_m.cpu().numpy(), ref_c.cpu().numpy()
    assert np.all(ref_c[:, 0] > 0) and np.all(ref_c[:, 2] > 0)
    for world in (1, 2, 3):
        for tile in (0, 7, 37):
            m = torch.zeros((5, 2, spp), dtype=torch.float64, device=ctx.device)
            c = torch.zeros((5, 3), dtype=torch.int64, device=ctx.device)
            for r in range(world):
                part = torch.zeros_like(m)
                sweep.mer_sweep_local(ctx, lp, cons, snrs, spp, TAPS4, rank=r, world=world, tile=tile, mer=part, counts=c, **kw)
                m += part
            ctx.sync()
            assert np.array_equal(m.cpu().numpy(), ref_m), (world, tile)
            assert np.array_equal(c.cpu().numpy(), ref_c), (world, tile)


def test_P1_ber_snr_figure_in_one_call():
    """`Task 3/Main_model_Task_3.m:192-268`: all four curves of the figure in one call, 2,048 streams per point, Task 3's
    scalar pilots 4/3 * max|constellation|."""
    sweep = _sweep()
    ctx = _ctx()
    p = OC.params_task4(alternate=False)
    lp = _lp(ctx, p)
    pts = [(c, float(snr), fig) for c in NAMES for snr, fig in RP.BER_SNR_FIGURE[c].items()]
    res = sweep.mer_sweep(ctx, lp, [c for c, _, _ in pts], [s for _, s, _ in pts], 2048, seed=21, pilot_scale=4.0 / 3.0)
    for k, (c, snr, fig) in enumerate(pts):
        assert abs(res["ber"][k] / fig - 1) < RP.ber_tolerance(fig, c), (c, snr, res["ber"][k], fig)


def test_P2_mer_at_25dB():
    """`Task 3/README.md:53-55`: MER 29.0341 dB and BER 0 at 25 dB (Np = 2, see reference_pins.P2)."""
    sweep = _sweep()
    ctx = _ctx()
    p = OC.params_task4(percent=0.25, alternate=False)
    lp = _lp(ctx, p)
    res = sweep.mer_sweep(ctx, lp, "16QAM", [25.0], 4096, seed=7, pilot_scale=4.0 / 3.0)
    assert abs(res["mer_db"][0] - RP.MER_AWGN_25DB) < 0.06, res["mer_db"]
    assert res["counts"][0, 0] == 0


def test_group_equals_single_context():
    from ofdm_b200 import Group
    sweep = _sweep()
    ctx = _ctx()
    p = OC.params_task4(alternate=False)
    lp = _lp(ctx, p)
    args = (["BPSK", "8PSK", "16QAM"], [3.0, 9.0, 15.0], 41, TAPS4)
    kw = dict(seed=3, tile=16, sto=[1, 0, 2], cfo=0.01, pilot_scale=4.0 / 3.0, near_eps=1e-3)
    m, c = sweep.mer_sweep_local(ctx, lp, *args, **kw)
    ctx.sync()
    with Group([0, 0]) as g:
        gm, gc = g.sweep_mer(lp, *args, **kw)
    assert np.array_equal(gm.view(np.int64), m.cpu().numpy().view(np.int64))
    assert np.array_equal(gc, c.cpu().numpy())


@pytest.mark.parametrize("layout", ["interleaved", "split"])
def test_mex_gateway_equals_c_call(layout):
    from test_gpu_mex import Mex
    sweep = _sweep()
    subprocess.run(["make", "-C", os.path.join(ROOT, "mex")], check=True, capture_output=True)
    mex = Mex(layout)
    ctx = _ctx()
    p = OC.params_task4(alternate=False)
    lp = _lp(ctx, p)
    try:
        args = [float(p.Nfft), float(p.T_Guard), float(p.N_carrier), float(p.N_symb), float(p.Amount_ODFM_SpF), p.Constellation,
                p.dataCarriers.astype(float), p.pilotCarriers.astype(float), p.pilotValues, O.DEFAULT_REGISTER.astype(float)]
        cons, snrs, spp = ["QPSK", "16QAM"], [6.0, 12.0], 33
        got_m, got_c = mex.call("sweep_mer", *args, np.array([2.0, 4.0]), np.asarray(snrs), float(spp), np.asarray(TAPS4, dtype=float), 3.0,
                                np.array([0.0, 4.0]), 0.02, 4.0 / 3.0, 1e-3, nout=2)
        res = sweep.mer_sweep(ctx, lp, cons, snrs, spp, TAPS4, seed=3, sto=[0, 4], cfo=0.02, pilot_scale=4.0 / 3.0, near_eps=1e-3)
        assert got_m.shape == (spp, 2 * len(snrs))
        assert np.array_equal(got_m.reshape(spp, 2, len(snrs), order="F").transpose(2, 1, 0), res["mer"])
        assert np.array_equal(got_c.astype(np.int64), res["counts"])
    finally:
        mex.lib.ofdm_mex_shim_exit()


def _raw_call(ctx, lp, mp):
    mer = torch.zeros(64, dtype=torch.float64, device=ctx.device)
    cnt = torch.zeros(16, dtype=torch.int64, device=ctx.device)
    return ctx.lib.ofdm_sweep_mer(ctx.h, C.byref(lp), C.byref(mp), ctx.p(mer), ctx.p(cnt))


def test_refusals():
    sweep = _sweep()
    ctx = _ctx()
    p = OC.params_task4(alternate=False)
    lp = _lp(ctx, p)
    c64 = _ctx("f64")
    assert _raw_call(c64, _lp(c64, p), sweep.mer_params("16QAM", [5.0], 4)) == -4          # OFDM_ERR_UNSUPPORTED
    assert "FP64" in c64.lib.ofdm_last_error(c64.h).decode()
    p4k = OC.params_task5(comb=4)
    assert _raw_call(ctx, _lp(ctx, p4k), sweep.mer_params("16QAM", [5.0], 4)) == -4
    assert "Nfft = 1024" in ctx.lib.ofdm_last_error(ctx.h).decode()
    bad = [(sweep.mer_params([9], [5.0], 4), "unknown constellation"),
           (sweep.mer_params("16QAM", [5.0], 4, sto=-1), "STO of point 0 is negative"),
           (sweep.mer_params(["QPSK", "BPSK"], [5.0, np.nan], 4), "SNR of point 1 is NaN"),
           (sweep.mer_params("16QAM", [5.0], 4, cfo=np.inf), "CFO of point 0 is not finite"),
           (sweep.mer_params("16QAM", [5.0], 4, rank=2, world=2), "rank must lie"),
           (sweep.mer_params("16QAM", [5.0], 4, taps=[[0.5, 1.0]]), "tap delays")]
    empty = sweep.mer_params("16QAM", [5.0], 4)
    empty.n_points = 0
    bad.append((empty, "at least one point"))
    for mp, text in bad:
        assert _raw_call(ctx, lp, mp) == -1                                                  # OFDM_ERR_INVALID
        msg = ctx.lib.ofdm_last_error(ctx.h).decode()
        assert "ofdm_sweep_mer" in msg and text in msg, msg
