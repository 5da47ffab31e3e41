"""GPU parity of the fused chains (TX, Task-5 channel, M1 RX chain) against the oracle's script-level
restatement, plus size-independent properties at larger batch."""
import numpy as np
import pytest

import oracle as O
from oracle import chains as OC

pytestmark = pytest.mark.gpu
TAPS5 = [[0, 1], [4, .8], [10, .6], [15, .4], [21, .2], [25, .1]]


@pytest.fixture(scope="module")
def G():
    import ofdm_b200
    return ofdm_b200


def rel_err(a, b):
    return np.linalg.norm((np.asarray(a) - np.asarray(b)).ravel()) / max(np.linalg.norm(np.asarray(b).ravel()), 1e-300)


def _lp(ctx, p, scramble=True):
    return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                           p.pilotCarriers, p.pilotValues, scramble=scramble)


PARAMS = {
    "t5_comb4": lambda: OC.params_task5(comb=4),
    "t5_comb7": lambda: OC.params_task5(comb=7),
    "t4": lambda: OC.params_task4(),
    "t4_8psk": lambda: OC.params_task4(Constellation="8PSK"),
    "t4_bpsk": lambda: OC.params_task4(Constellation="BPSK"),
}


@pytest.mark.parametrize("name", list(PARAMS))
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_tx_chain_matches_oracle(G, name, prec):
    p = PARAMS[name]()
    ctx = G.default_context(prec)
    lp = _lp(ctx, p)
    rng = np.random.default_rng(1)
    B = 3
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    tx = ctx.tx_chain(lp, ctx.bits(bits.ravel()), B).cpu().numpy().reshape(B, -1)
    for b in range(B):
        ref, _, _ = OC.tx_chain(p, bits[b])
        assert rel_err(tx[b], ref) < (1e-12 if prec == "f64" else 2e-6)


@pytest.mark.parametrize("name", list(PARAMS))
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_rx_chain_matches_oracle(G, name, prec):
    p = PARAMS[name]()
    ctx = G.default_context(prec)
    lp = _lp(ctx, p)
    rng = np.random.default_rng(2)
    B = 3
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    h, _ = O.get_MP_channel_resp(TAPS5, p.Nfft)
    normals = rng.standard_normal((B, 2, p.stream_len))
    rxs, refs = [], []
    for b in range(B):
        t, _, _ = OC.tx_chain(p, bits[b])
        r = OC.channel_task5(p, t, 18.0, TAPS5, normals=normals[b])
        rxs.append(r)
        refs.append(OC.rx_chain_task5(p, r, bits[b]))
    rx_d = ctx.cplx(np.stack(rxs).reshape(B, p.N_symb, p.Nfft + p.T_Guard))
    res = ctx.rx_chain_t5(lp, rx_d, B, tx_bits_dev=ctx.bits(bits.ravel()), near_eps=1e-3 if prec == "f32" else 1e-9, want_err_per_stream=True)
    ctx.sync()
    H = res["H"].cpu().numpy()
    got_bits = ctx.host_bits(res["bits"], B * p.stream_bits).reshape(B, -1)
    counts = res["counts"].cpu().numpy()
    eps = res["err_per_stream"].cpu().numpy()
    mism = 0
    for b in range(B):
        assert rel_err(H[b], refs[b]["H"]) < (1e-10 if prec == "f64" else 2e-5)
        mism += int(np.sum(got_bits[b] != refs[b]["bits"]))
        assert eps[b] == int(np.sum(got_bits[b] != bits[b]))
    ref_err = sum(r["errors"] for r in refs)
    assert counts[1] == B * p.stream_bits
    assert counts[0] == int(np.sum(got_bits != bits))
    if prec == "f64":
        assert mism == 0 and counts[0] == ref_err
    else:
        # FP32 decisions may differ only for symbols within epsilon of a boundary; each flips <= bps
        # decided bits, which the descrambler spreads to <= 3*bps
        assert mism <= 3 * p.bps * counts[2]
        assert abs(int(counts[0]) - ref_err) <= mism


def test_rx_chain_noise_free_loopback_ber_zero(G):
    """SURVEY KAT 3 through the fused chains at a larger batch: BER = 0 without impairments."""
    p = OC.params_task5(comb=4)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rng = np.random.default_rng(3)
    B = 64
    bits = rng.integers(0, 2, B * p.stream_bits).astype(np.uint8)
    bd = ctx.bits(bits)
    tx = ctx.tx_chain(lp, bd, B)
    res = ctx.rx_chain_t5(lp, tx, B, tx_bits_dev=bd)
    counts = res["counts"].cpu().numpy()
    assert counts[0] == 0 and counts[1] == B * p.stream_bits
    assert np.array_equal(ctx.host_bits(res["bits"], B * p.stream_bits), bits)
    H = res["H"].cpu().numpy()
    assert np.max(np.abs(H - 1)) < 1e-4


def test_channel_t5_device_matches_oracle_and_philox_is_batch_invariant(G):
    p = OC.params_task5(comb=4)
    ctx = G.default_context("f64")
    lp = _lp(ctx, p)
    rng = np.random.default_rng(4)
    B = 2
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    h, _ = O.get_MP_channel_resp(TAPS5, p.Nfft)
    normals = rng.standard_normal((B, 2, p.stream_len))
    tx = ctx.tx_chain(lp, ctx.bits(bits.ravel()), B)
    rx = ctx.channel_t5(tx, snr_db=20.0, h_dev=ctx.cplx(h), normals_dev=ctx.real(normals, ctx.rdtype)).cpu().numpy().reshape(B, -1)
    for b in range(B):
        t, _, _ = OC.tx_chain(p, bits[b])
        ref = OC.channel_task5(p, t, 20.0, TAPS5, normals=normals[b])
        assert rel_err(rx[b], ref) < 1e-12
    # counter-based noise: stream k gets the same realisation whatever the batch split
    c32 = G.default_context("f32")
    lp32 = _lp(c32, p)
    tx32 = c32.tx_chain(lp32, c32.bits(bits.ravel()), B)
    full = c32.channel_t5(tx32, snr_db=20.0, seed=77, first_stream_id=10).cpu().numpy()
    second = c32.channel_t5(tx32[1:2].contiguous(), snr_db=20.0, seed=77, first_stream_id=11).cpu().numpy()
    assert np.array_equal(full[1], second[0])


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_tx_power_handover_and_fused_channel_equals_two_step_channel(G, prec):
    """ofdm_tx_chain_p / ofdm_channel_t5_p: the TX stage measures sum |x|^2 (`Noise.m:3`) so the channel stage skips
    its own pass; and the fused Philox channel (tiles with carried history) equals add_noise -> apply_fir exactly."""
    import torch
    p = OC.params_task5(comb=4)
    ctx = G.default_context(prec)
    lp = _lp(ctx, p)
    rng = np.random.default_rng(11)
    B = 3
    bits = ctx.bits(rng.integers(0, 2, B * p.stream_bits).astype(np.uint8))
    tx0 = ctx.tx_chain(lp, bits, B)
    tx, psum = ctx.tx_chain(lp, bits, B, want_power=True)
    assert torch.equal(torch.view_as_real(tx), torch.view_as_real(tx0))
    t64 = tx.reshape(B, -1).to(torch.complex128)
    ref = (t64.real ** 2 + t64.imag ** 2).sum(dim=1)
    assert float(((psum - ref).abs() / ref).max()) < (1e-6 if prec == "f32" else 1e-12)
    hd = ctx.cplx(O.get_MP_channel_resp(TAPS5, p.Nfft)[0])
    own = ctx.channel_t5(tx, snr_db=12.0, h_dev=hd, seed=9, first_stream_id=5)
    handed = ctx.channel_t5(tx, snr_db=12.0, h_dev=hd, seed=9, first_stream_id=5, power_sum=psum)
    assert rel_err(handed.cpu().numpy(), own.cpu().numpy()) < (1e-6 if prec == "f32" else 1e-12)
    # two-step composition through the reference-named functions: Noise then conv+truncate (`Main_model_Task_5.m:108,123-127`)
    noisy = ctx.channel_t5(tx, snr_db=12.0, seed=9, first_stream_id=5)
    two_step = ctx.channel_t5(noisy, h_dev=hd)
    if prec == "f32":
        assert torch.equal(torch.view_as_real(own), torch.view_as_real(two_step))
    else:   # the FP64 kernels contract their multiply-adds differently
        assert rel_err(own.cpu().numpy(), two_step.cpu().numpy()) < 1e-14


@pytest.mark.parametrize("L,D", [(5001, 7), (100, 1), (2048, 26), (4097, 2), (20001, 300)])
def test_fused_channel_on_ragged_lengths_equals_two_step(G, L, D):
    """Tile edges of the fused AWGN + FIR kernel: odd and short streams, a single tap, a filter longer than a Philox
    pair run, chunk boundaries (8 tiles of 2,048) -- always bit-identical to Noise followed by conv+truncate in FP32."""
    import torch
    ctx = G.default_context("f32")
    rng = np.random.default_rng(L + D)
    B = 2
    x = ctx.cplx((rng.standard_normal((B, L)) + 1j * rng.standard_normal((B, L))))
    h = np.zeros(D, dtype=complex)
    nz = rng.choice(D, size=min(D, 5), replace=False)
    h[nz] = rng.standard_normal(len(nz)) + 1j * rng.standard_normal(len(nz))
    h[0] = 1.0
    hd = ctx.cplx(h)
    fused = ctx.channel_t5(x, snr_db=9.0, h_dev=hd, seed=3, first_stream_id=7)
    two_step = ctx.channel_t5(ctx.channel_t5(x, snr_db=9.0, seed=3, first_stream_id=7), h_dev=hd)
    assert torch.equal(torch.view_as_real(fused), torch.view_as_real(two_step))
    normals = ctx.real(rng.standard_normal((B, 2, L)), ctx.rdtype)
    fused_n = ctx.channel_t5(x, snr_db=9.0, h_dev=hd, normals_dev=normals)
    two_step_n = ctx.channel_t5(ctx.channel_t5(x, snr_db=9.0, normals_dev=normals), h_dev=hd)
    assert torch.equal(torch.view_as_real(fused_n), torch.view_as_real(two_step_n))


def test_rx_chain_host_entry(G):
    import torch
    p = OC.params_task5(comb=4)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rng = np.random.default_rng(5)
    B = 10
    bits = rng.integers(0, 2, B * p.stream_bits).astype(np.uint8)
    bd = ctx.bits(bits)
    tx = ctx.tx_chain(lp, bd, B)
    rx = ctx.channel_t5(tx, snr_db=15.0, h_dev=ctx.cplx(O.get_MP_channel_resp(TAPS5, p.Nfft)[0]), seed=5)
    dev = ctx.rx_chain_t5(lp, rx, B, tx_bits_dev=bd)
    ctx.sync()
    rx_h = rx.cpu().pin_memory()
    tb_h = bd.cpu().pin_memory()
    ob_h = torch.zeros_like(tb_h).pin_memory()
    H_h = torch.zeros((B, p.N_carrier), dtype=torch.complex64).pin_memory()
    counts = ctx.rx_chain_t5_host(lp, rx_h, B, tb_h, ob_h, H_h, chunk=4)   # 3 chunks, ragged last one
    dc = dev["counts"].cpu().numpy()
    assert counts[0] == dc[0] and counts[1] == dc[1]
    assert torch.equal(ob_h, dev["bits"].cpu()) and torch.equal(H_h, dev["H"].cpu())


@pytest.mark.parametrize("chain", ["task5", "task4"])
def test_sweep_counts_do_not_depend_on_the_split(G, chain):
    """SURVEY 4(iii): everything random is a Philox stream keyed by the global stream id => ofdm_sweep_ber returns identical
    counters for any rank count and any tile size."""
    from ofdm_b200 import sweep
    ctx = G.default_context("f32")
    if chain == "task5":
        p, taps, snrs, spp = OC.params_task5(comb=4), TAPS5, [4.0, 10.0, 16.0], 23
    else:
        p, taps, snrs, spp = OC.params_task4(), [[0, 1], [4, .6], [10, .3]], [8.0, 25.0], 21
    lp = _lp(ctx, p)
    one = sweep.ber_sweep(ctx, lp, snrs, spp, taps, chain, seed=3, tile=8)
    halves = sum(sweep.ber_sweep(ctx, lp, snrs, spp, taps, chain, seed=3, rank=r, world=2, tile=5) for r in range(2))
    eighths = sum(sweep.ber_sweep(ctx, lp, snrs, spp, taps, chain, seed=3, rank=r, world=8, tile=64) for r in range(8))
    assert np.array_equal(one, halves) and np.array_equal(one, eighths)
    assert np.all(one[:, 1] == spp * p.stream_bits)
    ber = one[:, 0] / one[:, 1]
    assert np.all(np.diff(ber) < 0) and 0.02 < ber[0] < 0.5
    other_seed = sweep.ber_sweep(ctx, lp, snrs, spp, taps, chain, seed=4, tile=8)
    assert not np.array_equal(one[:, 0], other_seed[:, 0])


def test_sweep_task5_equals_the_composed_calls(G):
    """ofdm_sweep_ber (chain 0) == ofdm_payload_bits -> DeScrambler -> ofdm_tx_chain_p -> ofdm_channel_t5_p -> ofdm_rx_chain_t5 with
    the same keys, each of which is compared with the oracle elsewhere in this file."""
    import torch
    from ofdm_b200 import sweep
    p = OC.params_task5(comb=4)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    snrs, spp, seed = [6.0, 12.0], 10, 11
    got = sweep.ber_sweep(ctx, lp, snrs, spp, TAPS5, "task5", seed=seed, tile=4, near_eps=1e-3)
    hd = ctx.cplx(O.get_MP_channel_resp(TAPS5, p.Nfft)[0])
    words = p.stream_bits // 32
    lp_raw = _lp(ctx, p, scramble=False)
    for i, snr in enumerate(snrs):
        sbits = torch.zeros(spp * words, dtype=torch.int32, device=ctx.device)
        ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(sbits), spp, words, seed, i * spp))
        # the sweep draws the SCRAMBLED frames s; the payload is p = DeScrambler(s), and the TX chain on p equals the chain on s
        # without its scrambler bit for bit (Scrambler(p) = s)
        bits = ctx.scramble(sbits, spp * p.Amount_OFDM_Frames, p.frame_bits, descramble=True)
        assert torch.equal(ctx.scramble(bits, spp * p.Amount_OFDM_Frames, p.frame_bits), sbits)
        tx, psum = ctx.tx_chain(lp, bits, spp, want_power=True)
        tx_raw = ctx.tx_chain(lp_raw, sbits, spp)
        assert torch.equal(torch.view_as_real(tx), torch.view_as_real(tx_raw))
        rx = ctx.channel_t5(tx, snr_db=snr, h_dev=hd, seed=seed, first_stream_id=i * spp, power_sum=psum)
        res = ctx.rx_chain_t5(lp, rx, spp, tx_bits_dev=bits, near_eps=1e-3)
        ctx.sync()
        assert np.array_equal(res["counts"].cpu().numpy(), got[i, :3]) and got[i, 3] == 0
    # the payload generator: uniform bits, distinct per stream, independent of how the range is cut
    b = torch.zeros(6 * words, dtype=torch.int32, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(b), 6, words, seed, 100))
    b2 = torch.zeros(2 * words, dtype=torch.int32, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(b2), 2, words, seed, 103))
    ctx.sync()
    assert torch.equal(b[3 * words:5 * words], b2)
    ones = np.unpackbits(b.cpu().numpy().view(np.uint8)).mean()
    assert abs(ones - 0.5) < 0.005 and not torch.equal(b[:words], b[words:2 * words])


def test_sweep_task4_against_oracle(G):
    """The CFO/STO leg of config 5: ofdm_sweep_ber (chain 1) against the ORACLE's Task-4 receiver run on the very streams the
    sweep builds (payload, Philox noise, STO / CFO draws rebuilt through the exported pieces with the sweep's keys)."""
    import torch
    from ofdm_b200 import sweep
    TAPS4 = [[0, 1], [4, .6], [10, .3]]
    p = OC.params_task4()
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    snrs, spp, seed = [18.0, 35.0], 8, 5
    got = sweep.ber_sweep(ctx, lp, snrs, spp, TAPS4, "task4", seed=seed, tile=5, near_eps=1e-3)
    good_total = 0
    words = p.stream_bits // 32
    hd = ctx.cplx(O.get_MP_channel_resp(TAPS4, p.Nfft)[0])
    for i, snr in enumerate(snrs):
        g0 = i * spp
        sbits = torch.zeros(spp * words, dtype=torch.int32, device=ctx.device)
        ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(sbits), spp, words, seed, g0))
        bits = ctx.scramble(sbits, spp * p.Amount_OFDM_Frames, p.frame_bits, descramble=True)       # payload p = DeScrambler(s)
        sto = torch.zeros(spp, dtype=torch.int32, device=ctx.device)
        cfo = torch.zeros(spp, dtype=torch.float64, device=ctx.device)
        ctx._chk(ctx.lib.ofdm_draw_sto_cfo(ctx.h, spp, seed, g0, p.Nfft + p.T_Guard, 30, ctx.p(sto), ctx.p(cfo)))
        tx = ctx.tx_chain(lp, bits, spp).reshape(spp, -1)
        noisy, _ = ctx.add_noise(tx, float(snr), seed=seed, first_stream_id=g0)
        rx = ctx.apply_fir(ctx.add_cfo(ctx.add_sto(noisy, sto), cfo, p.Nfft), hd)
        ctx.sync()
        sto_h, cfo_h = sto.cpu().numpy(), cfo.cpu().numpy()
        assert np.all((sto_h >= 0) & (sto_h <= 1152)) and np.all((cfo_h >= -0.5) & (cfo_h < 30.5))
        # the sweep is exactly the fused chain on these streams ...
        out = ctx.rx_chain_t4_fused(lp, rx.reshape(spp, p.N_symb, -1), tx_bits_dev=bits, near_eps=1e-3)
        ctx.sync()
        assert np.array_equal(out["counts"].cpu().numpy(), got[i, :3]) and int(out["fail"].sum()) == got[i, 3]
        assert got[i, 1] == spp * p.stream_bits
        # ... and the fused chain agrees with the oracle's receiver stream by stream
        bits_h = ctx.host_bits(bits, spp * p.stream_bits).reshape(spp, -1)
        got_bits = ctx.host_bits(out["bits"], spp * p.stream_bits).reshape(spp, -1)
        rx_h = rx.cpu().numpy().astype(np.complex128)
        tg, ifo, fail = out["TgPosition"].cpu().numpy(), out["IFO"].cpu().numpy(), out["fail"].cpu().numpy()
        mism, n_good = 0, 0
        for b in range(spp):
            try:
                ref = OC.rx_chain_task4(p, rx_h[b], bits_h[b])
            except IndexError:            # remove_IFO found no bin above 0.77: MATLAB errors, the device reports IFO = -1
                assert ifo[b] == -1
                continue
            assert tg[b] == ref["TgPosition"] and ifo[b] == ref["IFO"] and bool(fail[b]) == (ref["TgPosition"] == 65)
            if ref["errors"] < 0.05 * p.stream_bits:      # a stream the reference algorithm synchronised: decisions comparable
                mism += int(np.sum(got_bits[b] != ref["bits"]))
                n_good += 1
        good_total += n_good
        assert mism <= 3 * p.bps * int(got[i, 2])
    assert good_total >= 3        # the reference's own synchroniser fails on a good share of the STO/CFO draws (BER ~ 0.18 at 30 dB)


def test_sto_cfo_draws_are_uniform(G):
    import torch
    ctx = G.default_context("f32")
    n = 200000
    sto = torch.zeros(n, dtype=torch.int32, device=ctx.device)
    cfo = torch.zeros(n, dtype=torch.float64, device=ctx.device)
    ctx._chk(ctx.lib.ofdm_draw_sto_cfo(ctx.h, n, 9, 0, 1152, 30, ctx.p(sto), ctx.p(cfo)))
    ctx.sync()
    s, c = sto.cpu().numpy(), cfo.cpu().numpy()
    assert s.min() == 0 and s.max() == 1152 and abs(s.mean() - 576) < 3
    hist = np.bincount(s, minlength=1153)
    assert hist.min() > 100 and hist.max() < 260                   # mean 173.5 per value
    assert c.min() >= -0.5 and c.max() < 30.5 and abs(c.mean() - 15.0) < 0.08
    frac = (c + 0.5) % 1.0
    assert abs(frac.mean() - 0.5) < 0.005 and abs(np.corrcoef(s[:-1], s[1:])[0, 1]) < 0.01


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_rx_chain_task4_matches_oracle(G, prec):
    """Config 2 (M2): the whole Task-4 sync + CE chain, batched on the device, against the oracle per stream."""
    TAPS4 = [[0, 1], [4, .6], [10, .3]]
    p = OC.params_task4()
    ctx = G.default_context(prec)
    lp = _lp(ctx, p)
    rng = np.random.default_rng(8)
    cases = [(37, 7.24), (900, 0.24), (150, 12.4), (0, 0.0), (611, 3.3)]
    B = len(cases)
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    rxs, refs = [], []
    for b, (sto, cfo) in enumerate(cases):
        tx, _, _ = OC.tx_chain(p, bits[b], fast=True)
        rx = OC.impair_task4(p, tx, SNR_dB=28, Time_Delay=sto, Freq_Shift=cfo, taps=TAPS4, rng=rng)
        rxs.append(rx)
        refs.append(OC.rx_chain_task4(p, rx, bits[b]))
    out = ctx.rx_chain_t4(lp, ctx.cplx(np.stack(rxs)), tx_bits_dev=ctx.bits(bits.ravel()), near_eps=1e-3 if prec == "f32" else 1e-9)
    ctx.sync()
    tg = out["TgPosition"].cpu().numpy(); ifo = out["IFO"].cpu().numpy()
    fo = out["FreqOffset"].cpu().numpy(); tau = out["tau"].cpu().numpy(); ph = out["phase_shift"].cpu().numpy()
    got = ctx.host_bits(out["bits"], B * p.stream_bits).reshape(B, -1)
    mism = 0
    for b in range(B):
        assert tg[b] == refs[b]["TgPosition"] and ifo[b] == refs[b]["IFO"]
        tol = 1e-9 if prec == "f64" else 2e-5
        assert abs(fo[b] - refs[b]["FreqOffset"]) < tol and abs(tau[b] - refs[b]["tau"]) < tol
        assert abs(ph[b] - refs[b]["phase_shift"]) < (1e-7 if prec == "f64" else 2e-3)
        mism += int(np.sum(got[b] != refs[b]["bits"]))
    counts = out["counts"].cpu().numpy()
    assert counts[1] == B * p.stream_bits and counts[0] == int(np.sum(got != bits))
    if prec == "f64":
        assert mism == 0
    else:
        assert mism <= 3 * p.bps * out["near"]
    # the reference's own pass criterion (`Main_model_Task_4.m:367`)
    assert counts[0] / counts[1] < 0.2


def test_rx_chain_task4_fused_matches_oracle_and_composed(G):
    """The fused M2 entry (ofdm_rx_chain_t4) against the oracle and against the composed per-function chain."""
    TAPS4 = [[0, 1], [4, .6], [10, .3]]
    p = OC.params_task4()
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rng = np.random.default_rng(9)
    cases = [(37, 7.24), (900, 0.24), (150, 12.4), (0, 0.0), (611, 3.3), (1152, 30.4), (1, 0.49)]
    B = len(cases)
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    rxs, refs = [], []
    for b, (sto, cfo) in enumerate(cases):
        tx, _, _ = OC.tx_chain(p, bits[b], fast=True)
        rx = OC.impair_task4(p, tx, SNR_dB=28, Time_Delay=sto, Freq_Shift=cfo, taps=TAPS4, rng=rng)
        rxs.append(rx)
        refs.append(OC.rx_chain_task4(p, rx, bits[b]))
    rx_d = ctx.cplx(np.stack(rxs))
    bd = ctx.bits(bits.ravel())
    out = ctx.rx_chain_t4_fused(lp, rx_d, tx_bits_dev=bd, near_eps=1e-3, want_H=True)
    comp = ctx.rx_chain_t4(lp, rx_d, tx_bits_dev=bd, near_eps=1e-3)
    ctx.sync()
    got = ctx.host_bits(out["bits"], B * p.stream_bits).reshape(B, -1)
    got_c = ctx.host_bits(comp["bits"], B * p.stream_bits).reshape(B, -1)
    tg = out["TgPosition"].cpu().numpy(); ifo = out["IFO"].cpu().numpy()
    fo = out["FreqOffset"].cpu().numpy(); tau = out["tau"].cpu().numpy(); ph = out["phase_shift"].cpu().numpy()
    H = out["H"].cpu().numpy()
    mism = 0
    def close(a, b, tol):      # NaN is a legitimate result of the reference algorithm (mean of an empty selection)
        return (np.isnan(a) and np.isnan(b)) or abs(a - b) < tol
    n_nan = 0
    for b in range(B):
        assert tg[b] == refs[b]["TgPosition"] and ifo[b] == refs[b]["IFO"]
        assert close(fo[b], refs[b]["FreqOffset"], 2e-5) and close(tau[b], refs[b]["tau"], 2e-5) and close(ph[b], refs[b]["phase_shift"], 2e-3)
        Href = refs[b]["H"][:400]
        if np.all(np.isfinite(Href)):
            # phase_shift is a mean of wrapped angles (`fine_sync.m:47-52`): one pilot angle within rounding of +-pi
            # moves it by 2*pi/n_kept (1.8e-3 here), and H carries exp(j*phase_shift).  Compare H with that
            # (separately bounded) phase difference taken out.
            dphi = ph[b] - refs[b]["phase_shift"]
            assert np.linalg.norm(H[b] * np.exp(-1j * dphi) - Href) / np.linalg.norm(Href) < 1e-3
        else:
            n_nan += 1
            assert np.all(np.isnan(H[b].real))
        mism += int(np.sum(got[b] != refs[b]["bits"]))
    assert n_nan >= 1          # the (37, 7.24) case: no tau survives the 1e-3 mask -> NaN propagates as in MATLAB
    counts = out["counts"].cpu().numpy()
    assert counts[1] == B * p.stream_bits and counts[0] == int(np.sum(got != bits))
    assert mism <= 3 * p.bps * max(int(counts[2]), int(comp["near"]))
    assert int(np.sum(got != got_c)) <= 3 * p.bps * max(int(counts[2]), int(comp["near"]))
    # switches off: plain demodulation chain, BER 0 on a clean stream
    tx0, _, _ = OC.tx_chain(p, bits[0], fast=True)
    clean = ctx.rx_chain_t4_fused(lp, ctx.cplx(tx0[None]), tx_bits_dev=ctx.bits(bits[0]), time_desync=False, freq_desync=False, mp_desync=False)
    assert clean["counts"].cpu().numpy()[0] == 0


@pytest.mark.parametrize("ncar,con,near_eps", [(800, "16QAM", 1e-3), (400, "8PSK", 1e-3), (400, "QPSK", 0.0), (416, "16QAM", 0.0)])
def test_rx_chain_task4_fast_kernel_variants(G, monkeypatch, ncar, con, near_eps):
    """Template variants of the warp-per-symbol Task-4 kernel (unpruned second DFT for N_carrier > 416, generic
    constellations, near-boundary counting off) against the oracle and against the generic block-FFT kernel.  At N_carrier
    800 the stream has 5 frames: 10 need more shared memory than the fused kernel may take, and the generic one would run."""
    from kernel_witness import witness
    TAPS4 = [[0, 1], [4, .6], [10, .3]]
    frames = 5 if ncar > 416 else 10
    p = OC.LinkParams(Nfft=1024, N_carrier=ncar, T_Guard=128, Amount_OFDM_Frames=frames, Amount_ODFM_SpF=5, Constellation=con)
    p.pilotCarriers, p.dataCarriers = O.pilot_layout_percent(ncar, 15, 1024, last_gap=2)
    p.pilotValues, _ = OC.make_pilot_values(len(p.pilotCarriers), p.N_symb, con, 4.0 / 3.0, True)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rng = np.random.default_rng(21)
    cases = [(900, 0.24), (611, 3.3), (1, 0.49)]
    B = len(cases)
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    rxs, refs = [], []
    for b, (sto, cfo) in enumerate(cases):
        tx, _, _ = OC.tx_chain(p, bits[b], fast=True)
        rx = OC.impair_task4(p, tx, SNR_dB=30, Time_Delay=sto, Freq_Shift=cfo, taps=TAPS4, rng=rng)
        rxs.append(rx)
        refs.append(OC.rx_chain_task4(p, rx, bits[b]))
    rx_d = ctx.cplx(np.stack(rxs))
    bd = ctx.bits(bits.ravel())
    fast, kf = witness(lambda: ctx.rx_chain_t4_fused(lp, rx_d, tx_bits_dev=bd, near_eps=near_eps, want_H=True))
    got = ctx.host_bits(fast["bits"], B * p.stream_bits).reshape(B, -1)
    monkeypatch.setenv("OFDM_B200_NO_FAST", "1")
    slow, ks = witness(lambda: ctx.rx_chain_t4_fused(lp, rx_d, tx_bits_dev=bd, near_eps=1e-3, want_H=True))
    monkeypatch.delenv("OFDM_B200_NO_FAST")
    if kf is not None:             # None: no CUPTI, kernel identities are not observable
        rx = [k for k in kf + ks if k[0] in ("rx_t4_fast_kernel", "rx_t4_kernel")]
        assert rx == [("rx_t4_fast_kernel", (32 if ncar > 416 else 13, con == "16QAM", near_eps > 0)), ("rx_t4_kernel", ())], rx
    got_s = ctx.host_bits(slow["bits"], B * p.stream_bits).reshape(B, -1)
    near = max(int(slow["counts"].cpu().numpy()[2]), 1)
    checked = 0
    for b in range(B):
        def close(a, r, tol):      # NaN is a legitimate result of the reference algorithm (mean of an empty selection)
            return (np.isnan(a) and np.isnan(r)) or abs(a - r) < tol
        assert int(fast["TgPosition"][b]) == refs[b]["TgPosition"] and int(fast["IFO"][b]) == refs[b]["IFO"]
        assert close(float(fast["tau"][b]), refs[b]["tau"], 2e-5) and close(float(slow["tau"][b]), refs[b]["tau"], 2e-5)
        # phase_shift is a mean of wrapped angles (`fine_sync.m:47-52`): on a stream the reference itself fails to
        # synchronise (its pass criterion is BER < 0.2, `Main_model_Task_4.m:367`) the angles cover the circle and every
        # one within rounding of +-pi moves the mean by 2*pi/n -- such streams only have to agree on NaN-ness.
        ref_ber = np.mean(refs[b]["bits"] != bits[b])
        dph = float(fast["phase_shift"][b]) - refs[b]["phase_shift"]
        assert np.isnan(float(fast["phase_shift"][b])) == np.isnan(refs[b]["phase_shift"])
        if np.isnan(dph) or ref_ber >= 0.2 or abs(dph) >= 2e-3:
            assert np.isnan(dph) or ref_ber >= 0.2 or abs(dph) < 2e-2
            continue
        checked += 1
        Href = refs[b]["H"][:ncar]
        assert np.linalg.norm(fast["H"][b].cpu().numpy() * np.exp(-1j * dph) - Href) / np.linalg.norm(Href) < 1e-3
        assert int(np.sum(got[b] != refs[b]["bits"])) <= 3 * p.bps * near
        if abs(float(fast["phase_shift"][b]) - float(slow["phase_shift"][b])) < 1e-4:
            assert int(np.sum(got[b] != got_s[b])) <= 3 * p.bps * near
    assert checked >= 1
    c = fast["counts"].cpu().numpy()
    assert c[1] == B * p.stream_bits and c[0] == int(np.sum(got != bits)) and (near_eps > 0 or c[2] == 0)


def test_fused_kernels_are_deterministic_across_launches(G):
    """Race detector of last resort (compute-sanitizer is not available on the GPU pool): every fused kernel, launched
    repeatedly on the same inputs at a batch that fills the machine, must reproduce its outputs bit for bit."""
    import torch
    ctx = G.default_context("f32")
    rng = np.random.default_rng(77)
    p = OC.params_task5(comb=4)
    lp = _lp(ctx, p)
    B = 700                                            # more streams than resident CTAs: the persistent loops wrap around
    bits = ctx.bits(rng.integers(0, 2, B * p.stream_bits).astype(np.uint8))
    h, _ = O.get_MP_channel_resp(TAPS5, p.Nfft)
    hd = ctx.cplx(h)
    ref = None
    for rep in range(3):
        tx = ctx.tx_chain(lp, bits, B)
        rx = ctx.channel_t5(tx, snr_db=14.0, h_dev=hd, seed=4)
        res = ctx.rx_chain_t5(lp, rx, B, tx_bits_dev=bits, want_bits=True, want_H=True, near_eps=1e-3)
        cur = (tx.clone(), rx.clone(), res["bits"].clone(), torch.view_as_real(res["H"]).clone(), res["counts"].clone())
        if ref is None:
            ref = cur
        else:
            for a, b_ in zip(ref, cur):
                assert torch.equal(a, b_)
    assert int(ref[4][0]) > 0                          # 14 dB: there are errors to count
    p4 = OC.params_task4()
    lp4 = _lp(ctx, p4)
    B4 = 320
    t4, _, _ = OC.tx_chain(p4, rng.integers(0, 2, p4.stream_bits).astype(np.uint8), fast=True)
    base = OC.impair_task4(p4, t4, SNR_dB=28, Time_Delay=611, Freq_Shift=3.3, taps=[[0, 1], [4, .6], [10, .3]], rng=rng)
    rx4 = ctx.cplx(np.tile(base[None], (B4, 1)))
    rx4 = ctx.add_noise(rx4, 30.0, seed=9)[0]          # distinct streams
    ref4 = None
    for rep in range(3):
        r = ctx.rx_chain_t4_fused(lp4, rx4, near_eps=1e-3, want_H=True)
        cur = (r["bits"].clone(), torch.view_as_real(r["H"]).clone(), r["tau"].clone(), r["phase_shift"].clone(), r["TgPosition"].clone(), r["counts"].clone())
        if ref4 is None:
            ref4 = cur
        else:
            for a, b_ in zip(ref4, cur):
                assert torch.equal(a, b_) or (a.is_floating_point() and torch.equal(torch.nan_to_num(a), torch.nan_to_num(b_)))


def test_persistent_wraparound_against_oracle(G):
    """B = 640 streams > 2 x 148 (tx4096) and > 3 x 148 (three-CTA rx4096) persistent CTAs: CTAs walk on to a second stream, so the
    prefetch cursor's stream-to-stream hop (`pf_advance`) and the per-stream state resets are compared with the oracle --
    TX samples, channel output with imported normals, channel estimate, decided bits and per-stream error counts, for all
    640 streams (the oracle's vectorised scrambler forms are bit-identical to its loops, `test_oracle_kats`)."""
    import torch
    p = OC.params_task5(comb=4)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rng = np.random.default_rng(640)
    B = 640
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    normals = rng.standard_normal((B, 2, p.stream_len)).astype(np.float32)
    bd = ctx.bits(bits.ravel())
    tx = ctx.tx_chain(lp, bd, B)
    hd = ctx.cplx(O.get_MP_channel_resp(TAPS5, p.Nfft)[0])
    rx = ctx.channel_t5(tx, snr_db=14.0, h_dev=hd, normals_dev=torch.from_numpy(normals).to(ctx.device))
    eps_near = 1e-3
    res = ctx.rx_chain_t5(lp, rx, B, tx_bits_dev=bd, near_eps=eps_near, want_err_per_stream=True)
    ctx.sync()
    tx_h = tx.cpu().numpy().reshape(B, -1)
    rx_h = rx.cpu().numpy().reshape(B, -1)
    H = res["H"].cpu().numpy()
    got = ctx.host_bits(res["bits"], B * p.stream_bits).reshape(B, -1)
    eps = res["err_per_stream"].cpu().numpy()
    counts = res["counts"].cpu().numpy()
    mism, ref_err = 0, 0
    for b in range(B):
        t, _, _ = OC.tx_chain(p, bits[b], fast=True)
        assert rel_err(tx_h[b], t) < 2e-6, b
        r = OC.channel_task5(p, t, 14.0, TAPS5, normals=normals[b].astype(np.float64))
        assert rel_err(rx_h[b], r) < 2e-6, b
        ref = OC.rx_chain_task5(p, r, bits[b], fast=True)
        assert rel_err(H[b], ref["H"]) < 2e-5, b
        assert eps[b] == int(np.sum(got[b] != bits[b])), b
        mism += int(np.sum(got[b] != ref["bits"]))
        ref_err += ref["errors"]
    assert counts[1] == B * p.stream_bits and counts[0] == int(eps.sum())
    assert mism <= 3 * p.bps * counts[2]
    assert abs(int(counts[0]) - ref_err) <= mism


def test_rx_chain_task4_split_path_matches_fused_and_oracle(G, monkeypatch):
    """Batches of 512 streams and more run the Task-4 chain as three kernels (t4_ifo / t4_sym / t4_post) instead of the fused
    persistent one: same integer estimates, same decisions up to near-boundary symbols, against the fused kernel for every
    stream and against the oracle for the distinct cases."""
    TAPS4 = [[0, 1], [4, .6], [10, .3]]
    p = OC.params_task4()
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rng = np.random.default_rng(19)
    cases = [(37, 7.24), (900, 0.24), (150, 12.4), (0, 0.0), (611, 3.3), (1152, 30.4), (1, 0.49), (77, 21.7)]
    bits = rng.integers(0, 2, (len(cases), p.stream_bits)).astype(np.uint8)
    rxs, refs = [], []
    for b, (sto, cfo) in enumerate(cases):
        tx, _, _ = OC.tx_chain(p, bits[b], fast=True)
        rx = OC.impair_task4(p, tx, SNR_dB=28, Time_Delay=sto, Freq_Shift=cfo, taps=TAPS4, rng=rng)
        rxs.append(rx)
        refs.append(OC.rx_chain_task4(p, rx, bits[b]))
    B = 520                                              # 65 copies of the eight cases: >= 512 selects the split path
    reps = B // len(cases)
    rx_d = ctx.cplx(np.tile(np.stack(rxs), (reps, 1)))
    bd = ctx.bits(np.tile(bits, (reps, 1)).ravel())
    l0 = ctx.launches
    split = ctx.rx_chain_t4_fused(lp, rx_d, tx_bits_dev=bd, near_eps=1e-3, want_H=True)
    ctx.sync()
    n_split = ctx.launches - l0
    monkeypatch.setenv("OFDM_B200_T4_FUSED", "1")
    l0 = ctx.launches
    fused = ctx.rx_chain_t4_fused(lp, rx_d, tx_bits_dev=bd, near_eps=1e-3, want_H=True)
    ctx.sync()
    assert n_split == 4 + 3 and ctx.launches - l0 == 4 + 1          # autocorrelation (2 + gated 2) + ifo / sym / post vs one fused kernel
    for key in ("TgPosition", "IFO", "fail"):
        assert np.array_equal(split[key].cpu().numpy(), fused[key].cpu().numpy()), key
    ts, tf = split["tau"].cpu().numpy(), fused["tau"].cpu().numpy()
    ok = np.isfinite(tf)
    assert np.array_equal(np.isfinite(ts), ok) and np.max(np.abs(ts[ok] - tf[ok])) < 1e-6
    gs = ctx.host_bits(split["bits"], B * p.stream_bits).reshape(B, -1)
    gf = ctx.host_bits(fused["bits"], B * p.stream_bits).reshape(B, -1)
    near = int(split["counts"][2].item()) + int(fused["counts"][2].item())
    assert int(np.sum(gs != gf)) <= 3 * p.bps * near
    for b in range(len(cases)):
        assert np.array_equal(gs[b], gs[b + 8 * (reps - 1)])                                  # copies decode alike
        assert split["TgPosition"][b].item() == refs[b]["TgPosition"] and split["IFO"][b].item() == refs[b]["IFO"]
    mism = sum(int(np.sum(gs[b] != refs[b]["bits"])) for b in range(len(cases)) if np.all(np.isfinite(refs[b]["H"][:400])))
    assert mism * reps <= 3 * p.bps * int(split["counts"][2].item())


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_channel_t4_fused_is_bit_identical_to_the_composition(G, prec):
    """ofdm_channel_t4_p (Noise -> add_STO -> add_CFO -> multipath in one pass, `Task 4/Main_model_Task_4.m:95,103,110,263-264`)
    against ofdm_add_noise / ofdm_add_sto / ofdm_add_cfo / ofdm_apply_fir called in turn: the same bits, for Philox and for
    imported normals, odd / even / negative / out-of-range offsets, a stream length that is no multiple of the tile."""
    import torch
    ctx = G.Context(0, prec)
    rng = np.random.default_rng(3)
    B, L, Nfft = 9, 2 * 16384 + 2 * 2048 + 777, 1024
    x = ctx.cplx(rng.standard_normal((B, L)) + 1j * rng.standard_normal((B, L)))
    sto = np.array([0, 1, 2, 611, 1152, -3, -40, L + 5, 777], dtype=np.int32)
    cfo = np.array([0.0, 0.24, -0.5, 3.3, 30.4, 12.5, 7.0, 1.0, 29.99])
    h = np.zeros(11); h[0], h[4], h[10] = 1.0, 0.6, 0.3
    hd = ctx.cplx(h.astype(complex))
    snr = np.linspace(5.0, 30.0, B)
    for normals in (None, ctx.real(rng.standard_normal((B, 2, L)), ctx.rdtype)):
        noisy, _ = ctx.add_noise(x, snr, normals_dev=normals, seed=11, first_stream_id=40)
        ref = ctx.apply_fir(ctx.add_cfo(ctx.add_sto(noisy, sto), cfo, Nfft), hd)
        got = ctx.channel_t4(x, snr, sto, cfo, Nfft, hd, normals_dev=normals, seed=11, first_stream_id=40)
        ctx.sync()
        assert torch.equal(torch.view_as_real(got), torch.view_as_real(ref))
    one = ctx.cplx(np.ones(1, dtype=complex))
    got = ctx.channel_t4(x, snr, sto, cfo, Nfft, one, seed=11, first_stream_id=40)
    ref = ctx.add_cfo(ctx.add_sto(ctx.add_noise(x, snr, seed=11, first_stream_id=40)[0], sto), cfo, Nfft)
    ctx.sync()
    assert torch.equal(torch.view_as_real(got), torch.view_as_real(ref))
    # the rotation itself against the oracle's add_CFO (double): FP32 1e-6 of the sample, FP64 1e-12
    got = ctx.add_cfo(x, cfo, Nfft).cpu().numpy()
    want = np.stack([O.add_CFO(x[b].cpu().numpy(), cfo[b], Nfft) for b in range(B)])
    assert np.max(np.abs(got - want)) < (2e-6 if prec == "f32" else 1e-11)


def test_rx4096_three_cta_kernel_against_the_two_cta_kernel(G, monkeypatch):
    """The three-CTA (`SLIM`) instantiation of rx4096_kernel -- one landing buffer, L2 prefetch, two-factor twiddles -- against
    the two-CTA one on 1,000 streams (CTAs of both walk over two or three streams): channel estimates to FP32 tolerance, the
    same error counts per stream except where a symbol sits within the counted near-boundary margin."""
    p = OC.params_task5(comb=4)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    B = 1000
    import torch
    g = torch.Generator(device=ctx.device); g.manual_seed(5)
    bd = torch.randint(-2**31, 2**31 - 1, (B * p.stream_bits // 32,), dtype=torch.int32, device=ctx.device, generator=g)
    tx, ps = ctx.tx_chain(lp, bd, B, want_power=True)
    rx = ctx.channel_t5(tx, snr_db=13.0, h_dev=ctx.cplx(O.get_MP_channel_resp(TAPS5, p.Nfft)[0]), seed=3, power_sum=ps)
    l0 = ctx.launches
    slim = ctx.rx_chain_t5(lp, rx, B, tx_bits_dev=bd, near_eps=1e-3, want_err_per_stream=True)
    ctx.sync()
    monkeypatch.setenv("OFDM_B200_NO_SLIM", "1")
    two = ctx.rx_chain_t5(lp, rx, B, tx_bits_dev=bd, near_eps=1e-3, want_err_per_stream=True)
    ctx.sync()
    assert ctx.launches - l0 == 2
    Hs, Ht = slim["H"].cpu().numpy(), two["H"].cpu().numpy()
    assert np.max(np.abs(Hs - Ht)) < 2e-6 * np.max(np.abs(Ht))
    cs, ct = slim["counts"].cpu().numpy(), two["counts"].cpu().numpy()
    assert cs[1] == ct[1] == B * p.stream_bits and cs[0] > 0
    bs = ctx.host_bits(slim["bits"], B * p.stream_bits)
    bt = ctx.host_bits(two["bits"], B * p.stream_bits)
    assert int(np.sum(bs != bt)) <= p.bps * int(cs[2] + ct[2])
    es, et = slim["err_per_stream"].cpu().numpy(), two["err_per_stream"].cpu().numpy()
    assert int(es.sum()) == cs[0] and int(et.sum()) == ct[0] and int(np.sum(np.abs(es - et))) <= p.bps * int(cs[2] + ct[2])


@pytest.mark.parametrize("ncar,tg,con", [(400, 128, "16QAM"), (1000, 256, "QPSK"), (100, 0, "8PSK"), (416, 64, "BPSK")])
def test_tx1024_fast_kernel_variants(G, monkeypatch, ncar, tg, con):
    """The warp-per-symbol TX kernel of the Nfft = 1024 shape (`tx1024_kernel`) on other carrier counts (up to 32 carrier
    groups per lane), guard lengths and constellations: against the oracle's TX chain, against the generic kernel, and
    scrambling inside the kernel against ofdm_scramble followed by the kernel without it (bit-identical)."""
    import torch
    p = OC.LinkParams(Nfft=1024, N_carrier=ncar, T_Guard=tg, Amount_OFDM_Frames=4, Amount_ODFM_SpF=3, Constellation=con)
    p.pilotCarriers, p.dataCarriers = O.pilot_layout_percent(p.N_carrier, 15, p.Nfft, last_gap=2)
    p.pilotValues, _ = OC.make_pilot_values(len(p.pilotCarriers), p.N_symb, p.Constellation, 4 / 3, True)
    ctx = G.default_context("f32")
    lp, lp_raw = _lp(ctx, p), _lp(ctx, p, scramble=False)
    rng = np.random.default_rng(ncar + tg)
    B = 5
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    bd = ctx.bits(bits.ravel())
    l0 = ctx.launches
    tx, ps = ctx.tx_chain(lp, bd, B, want_power=True)
    ctx.sync()
    assert ctx.launches - l0 == 2                       # tx1024_kernel + the ordered sum of its per-symbol power partials
    tx_h = tx.cpu().numpy().reshape(B, -1)
    for b in range(B):
        ref, _, _ = OC.tx_chain(p, bits[b], fast=True)
        assert rel_err(tx_h[b], ref) < 2e-6, b
        assert abs(ps[b].item() / np.sum(np.abs(ref) ** 2) - 1) < 1e-5
    if p.stream_bits % 32 == 0 and p.frame_bits >= 15:
        sb = ctx.scramble(bd, B * p.Amount_OFDM_Frames, p.frame_bits) if p.frame_bits % 32 == 0 else None
        if sb is not None:
            assert torch.equal(torch.view_as_real(ctx.tx_chain(lp_raw, sb, B)), torch.view_as_real(tx))
    monkeypatch.setenv("OFDM_B200_NO_FAST", "1")
    gen = ctx.tx_chain(lp, bd, B).cpu().numpy().reshape(B, -1)
    assert rel_err(gen, tx_h) < 2e-6


def test_channel_t4_long_impulse_response_and_short_streams(G):
    """ofdm_channel_t4_p at the corners of its staging: an impulse response as long as a third of a tile (history regenerated
    through the per-sample path), streams shorter than one tile, one stream -- still the bits of the four calls."""
    import torch
    ctx = G.default_context("f32")
    rng = np.random.default_rng(8)
    for B, L, D in ((1, 777, 300), (3, 2048, 700), (2, 2049, 1), (4, 5000, 1024)):
        x = ctx.cplx(rng.standard_normal((B, L)) + 1j * rng.standard_normal((B, L)))
        h = rng.standard_normal(D) * (rng.random(D) < 0.2)
        h[0] = 1.0
        hd = ctx.cplx(h.astype(complex))
        sto = rng.integers(-50, 400, B).astype(np.int32)
        cfo = rng.random(B) * 20 - 0.5
        ref = ctx.apply_fir(ctx.add_cfo(ctx.add_sto(ctx.add_noise(x, 12.0, seed=2, first_stream_id=9)[0], sto), cfo, 1024), hd)
        got = ctx.channel_t4(x, 12.0, sto, cfo, 1024, hd, seed=2, first_stream_id=9)
        ctx.sync()
        assert torch.equal(torch.view_as_real(got), torch.view_as_real(ref)), (B, L, D)


def test_rx4096_unaligned_frames_at_a_large_batch(G):
    """comb 7 (frames of 24,556 bits, streams of 49,112: neither ends on a word): 500 streams through the fast kernels -- stream
    and frame boundaries fall inside words of the packed bit arrays that two CTAs write -- loop-back without impairments must
    return every bit, and with noise the per-stream error counts must add up to the counter."""
    p = OC.params_task5(comb=7)
    assert p.frame_bits % 32 != 0 and p.stream_bits % 32 != 0
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    rng = np.random.default_rng(7)
    B = 500
    bits = rng.integers(0, 2, B * p.stream_bits).astype(np.uint8)
    bd = ctx.bits(bits)
    tx = ctx.tx_chain(lp, bd, B)
    l0 = ctx.launches
    res = ctx.rx_chain_t5(lp, tx, B, tx_bits_dev=bd, want_err_per_stream=True)
    ctx.sync()
    assert ctx.launches - l0 == 1                       # the fast kernel, not the generic one
    counts = res["counts"].cpu().numpy()
    assert counts[0] == 0 and counts[1] == B * p.stream_bits
    assert np.array_equal(ctx.host_bits(res["bits"], B * p.stream_bits), bits)
    rx = ctx.channel_t5(tx, snr_db=12.0, h_dev=ctx.cplx(O.get_MP_channel_resp(TAPS5, p.Nfft)[0]), seed=4)
    res = ctx.rx_chain_t5(lp, rx, B, tx_bits_dev=bd, want_err_per_stream=True)
    ctx.sync()
    got = ctx.host_bits(res["bits"], B * p.stream_bits)
    counts = res["counts"].cpu().numpy()
    eps = res["err_per_stream"].cpu().numpy()
    per_stream = (got != bits).reshape(B, -1).sum(axis=1)
    assert counts[0] == per_stream.sum() > 0 and np.array_equal(eps, per_stream)


def test_dynamic_stream_claims_give_the_bits_of_the_static_stride(G, monkeypatch):
    """rx4096 (three-CTA) and tx4096 claim their streams from a per-launch counter; which CTA processes a stream must not
    matter: 1,000 streams, every output bit-identical to the static-stride schedule."""
    import torch
    p = OC.params_task5(comb=4)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    B = 1000
    g = torch.Generator(device=ctx.device); g.manual_seed(11)
    bd = torch.randint(-2**31, 2**31 - 1, (B * p.stream_bits // 32,), dtype=torch.int32, device=ctx.device, generator=g)
    hd = ctx.cplx(O.get_MP_channel_resp(TAPS5, p.Nfft)[0])

    def run():
        tx, ps = ctx.tx_chain(lp, bd, B, want_power=True)
        rx = ctx.channel_t5(tx, snr_db=12.0, h_dev=hd, seed=3, power_sum=ps)
        res = ctx.rx_chain_t5(lp, rx, B, tx_bits_dev=bd, near_eps=1e-3, want_err_per_stream=True)
        ctx.sync()
        return tx, ps, res

    tx_d, ps_d, dyn = run()
    monkeypatch.setenv("OFDM_B200_STATIC_STREAMS", "1")
    tx_s, ps_s, sta = run()
    assert torch.equal(torch.view_as_real(tx_d), torch.view_as_real(tx_s)) and torch.equal(ps_d, ps_s)
    for key in ("bits", "H", "counts", "err_per_stream"):
        a, b = dyn[key], sta[key]
        assert torch.equal(torch.view_as_real(a) if a.is_complex() else a, torch.view_as_real(b) if b.is_complex() else b), key
    assert int(dyn["counts"][0]) > 0
