"""Every instantiation of the Nfft-4096 receiver (`rx4096_kernel<QAM16, NEAR, MASK, SLIM>`) and transmitter (`tx4096_kernel`), and
the fallbacks to the generic kernels, against the float64 oracle: layouts and CTA variants, frame geometries at the edges of
the kernels' loops, carrier counts and guards, batch sizes around the persistent grids, the near-boundary counter, optional
outputs, per-symbol pilot columns and scrambler registers whose cells 13 and 14 are set.

Which kernel ran is read from the CUDA activity of `torch.profiler` (one launch of `rx4096_kernel` and one of `rx_chain_kernel`
look alike to a launch counter); a box without CUPTI skips those asserts and still runs the parity ones."""
import ctypes as C

import numpy as np
import pytest

import oracle as O
from oracle import chains as OC
from kernel_witness import Registry, t4_phase_bounds as _t4_phase_bounds, witness as _witness

pytestmark = pytest.mark.gpu
TAPS5 = [[0, 1], [4, .8], [10, .6], [15, .4], [21, .2], [25, .1]]
# a scrambler register with cells 13 and 14 set: both taps of the pre-history fold (`Scrambler.m:18-28`) are exercised
REG = np.array([1, 1, 0, 1, 0, 0, 1, 1, 1, 0, 0, 1, 1, 1, 1], dtype=np.uint8)
SNR = {"BPSK": 0.0, "QPSK": 3.0, "8PSK": 7.0, "16QAM": 9.0}
# Decided bits may differ from the oracle only in symbols whose float64 margin (second-smallest minus smallest squared distance)
# is below this: the FP32 equalised symbols are within ~1e-5 of the oracle's (H to 2e-5 relative), a hundred times less.
BIT_SLACK_MARGIN = 1e-3
# counts[2] must lie between the oracle's counts at near_eps * (1 -+ NEAR_DELTA).  The FP32 margin of a unit-power symbol is off
# by about 2 * |c1 - c2| * |e_fp32 - e_oracle| <= 4 * 2e-6 = 8e-6 for the worst symbols seen (FFT and spline rounding,
# 1e-6 .. 2e-6 of |e|), i.e. below 1e-2 of near_eps = 1e-3.
NEAR_DELTA = 1e-2


@pytest.fixture(scope="module")
def G():
    import ofdm_b200
    return ofdm_b200


def rel_err(a, b):
    return np.linalg.norm((np.asarray(a) - np.asarray(b)).ravel()) / max(np.linalg.norm(np.asarray(b).ravel()), 1e-300)


def _lp(ctx, p, scramble=True):
    return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                           p.pilotCarriers, p.pilotValues, Register=p.Register, scramble=scramble)


def _link(comb=None, Nc=1024, Tg=512, SpF=7, frames=2, con="16QAM", reg=False, Nfft=4096):
    """Task-5 shape with a comb layout (`1:comb:N_carrier`) or, without comb, the percent-style layout of Tasks 1-4."""
    p = OC.LinkParams(Nfft=Nfft, N_carrier=Nc, T_Guard=Tg, Amount_OFDM_Frames=frames, Amount_ODFM_SpF=SpF, Constellation=con)
    if comb:
        p.pilotCarriers, p.dataCarriers = O.pilot_layout_comb(Nc, comb)
    else:
        p.pilotCarriers, p.dataCarriers = O.pilot_layout_percent(Nc, 15, Nfft, last_gap=2)
    p.pilotValues, _ = OC.make_pilot_values(len(p.pilotCarriers), p.N_symb, con, 2.0, True)
    if reg:
        p.Register = REG.copy()
    return p


def _random_pilots(p, rng, scale=2.0, jitter=0.3):
    """Np x S pilot values with a distinct random column per symbol: random phases, amplitudes within 1 -+ jitter of
    scale * max|dictionary|."""
    d, _ = O.constellation_func(p.Constellation)
    shape = (len(p.pilotCarriers), p.N_symb)
    amp = scale * np.max(np.abs(d)) * rng.uniform(1 - jitter, 1 + jitter, shape)
    p.pilotValues = amp * np.exp(1j * rng.uniform(-np.pi, np.pi, shape))
    assert not np.allclose(p.pilotValues[:, :1], p.pilotValues)
    return p


def _streams(p, B, seed, scramble=True):
    """B random payloads through the oracle's TX chain and Task-5 channel, rounded to the FP32 samples the kernels read."""
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    rx = np.empty((B, p.stream_len), dtype=np.complex64)
    for b in range(B):
        t, _, _ = OC.tx_chain(p, bits[b], scramble=scramble, fast=True)
        rx[b] = OC.channel_task5(p, t, SNR[p.Constellation], TAPS5, normals=rng.standard_normal((2, p.stream_len)))
    return bits, rx


# ------------------------------------------------------------------------------------------------------------- kernel witness
_W = Registry()                  # kernels seen, RX matrix cases that ran


CHAIN_KERNELS = ("rx4096_kernel", "rx_chain_kernel", "tx4096_kernel", "tx_chain_kernel", "tx1024_kernel")


def _expect(kernels, want, case):
    """The chain kernel that ran must be exactly `want` (one launch); records what was seen for the coverage test."""
    if not _W.record(kernels, case):
        return
    chain = [k for k in kernels if k[0] in CHAIN_KERNELS]
    assert chain == [want], f"{case}: expected {want}, the profiler saw {kernels}"


def K(q16, near, mask, slim):
    return ("rx4096_kernel", (q16, near, mask, slim))


GEN_RX = ("rx_chain_kernel", ("float",))
TX4096 = ("tx4096_kernel", ())


# ------------------------------------------------------------------------------------------------------------- checks
def _check_stream(p, got, ref, scramble=True):
    """Decided bits of one stream against the oracle: raw (pre-descrambler) bits may differ only inside symbols whose float64
    margin is below BIT_SLACK_MARGIN (each such symbol <= bps raw bits, <= 3 bps descrambled bits)."""
    raw = OC.scramble_frames(p, got, fast=True) if scramble else got
    flipped = np.unique(np.flatnonzero(raw != ref["raw_bits"]) // p.bps)
    if flipped.size:
        m = O.near_margin(ref["rx_iq"][flipped], p.Constellation)
        assert np.all(m < BIT_SLACK_MARGIN), f"decisions differ at margins {np.sort(m)[-3:]}"
    assert int(np.sum(got != ref["bits"])) <= 3 * p.bps * flipped.size


def _check_rx(ctx, p, res, refs, bits, near_eps, scramble=True):
    B = bits.shape[0]
    got = ctx.host_bits(res["bits"], B * p.stream_bits).reshape(B, -1)
    counts = res["counts"].cpu().numpy()
    eps = res["err_per_stream"].cpu().numpy()
    H = res["H"].cpu().numpy()
    lo = hi = 0
    for b in range(B):
        assert rel_err(H[b], refs[b]["H"]) < 2e-5, b
        _check_stream(p, got[b], refs[b], scramble)
        assert eps[b] == int(np.sum(got[b] != bits[b])), b
        m = O.near_margin(refs[b]["rx_iq"], p.Constellation)       # data carriers only
        lo += int(np.sum(m < near_eps * (1 - NEAR_DELTA)))
        hi += int(np.sum(m < near_eps * (1 + NEAR_DELTA)))
    assert counts[1] == B * p.stream_bits
    assert counts[0] == int(np.sum(got != bits)) == int(eps.sum())
    if near_eps > 0:
        assert lo <= counts[2] <= hi, (lo, int(counts[2]), hi)
    else:
        assert counts[2] == 0


# ------------------------------------------------------------------------------------------------------------- RX matrix
# id: (link parameters, options, expected kernel).  Options: near (near_eps), two (OFDM_B200_NO_SLIM), scramble,
# rx_offset (rx one sample past a 16-byte boundary), tx_offset (tx_bits 4 bytes past one).
RX_CASES = {
    # comb 4 -> MASK 0x1111
    "c4_three_near_reg": (dict(comb=4, reg=True), dict(near=1e-3), K(True, True, 0x1111, True)),
    "c4_three_1344w": (dict(comb=4, SpF=14), dict(), K(True, False, 0x1111, True)),                 # frames > 1,024 words
    "c4_two_1344w_near_reg": (dict(comb=4, SpF=14, reg=True), dict(near=1e-3, two=True), K(True, True, 0x1111, False)),
    "c4_two_spf1_tg0": (dict(comb=4, SpF=1, frames=3, Tg=0), dict(two=True), K(True, False, 0x1111, False)),
    "c4_three_2496w_s_eq_spf": (dict(comb=4, SpF=26, frames=1), dict(near=1e-3), K(True, True, 0x1111, True)),   # largest fast frame
    "c4_two_2496w_s_eq_spf": (dict(comb=4, SpF=26, frames=1, reg=True), dict(two=True), K(True, False, 0x1111, False)),
    "c4_nc1000_375w": (dict(comb=4, Nc=1000, SpF=4, reg=True), dict(near=1e-3), K(True, True, 0x1111, True)),     # frame_words % 4 = 3
    "c4_txbits_offset4": (dict(comb=4), dict(near=1e-3, tx_offset=True), K(True, True, 0x1111, True)),
    # comb 8 -> MASK 0x0101
    "c8_three_near_tg2": (dict(comb=8, Tg=2), dict(near=1e-3), K(True, True, 0x0101, True)),
    "c8_three_noscr": (dict(comb=8), dict(scramble=False), K(True, False, 0x0101, True)),
    "c8_two_near_reg": (dict(comb=8, reg=True), dict(near=1e-3, two=True), K(True, True, 0x0101, False)),
    "c8_two_tg0": (dict(comb=8, Tg=0), dict(two=True), K(True, False, 0x0101, False)),
    # MASK 0: comb 16 (aligned frames), comb 7 (frames of 24,556 bits), percent-style layouts
    "c16_three_near": (dict(comb=16), dict(near=1e-3), K(True, True, 0, True)),
    "c7_three_reg": (dict(comb=7, reg=True), dict(), K(True, False, 0, True)),
    "c16_two_tg0_reg": (dict(comb=16, Tg=0, reg=True), dict(two=True), K(True, False, 0, False)),
    "c7_two_near_noscr": (dict(comb=7), dict(near=1e-3, two=True, scramble=False), K(True, True, 0, False)),
    "p600_three_near_tg2": (dict(Nc=600, Tg=2), dict(near=1e-3), K(True, True, 0, True)),
    "p1000_three_1040w_tg0": (dict(Nc=1000, SpF=10, Tg=0, reg=True), dict(), K(True, False, 0, True)),
    "p1024_two_1065w_near": (dict(Nc=1024, SpF=10), dict(near=1e-3, two=True), K(True, True, 0, False)),
    # other constellations: rx4096_kernel<false, NEAR, 0, false>
    "bpsk_p1000_tg0_near_reg": (dict(con="BPSK", Nc=1000, Tg=0, reg=True), dict(near=1e-3), K(False, True, 0, False)),
    "qpsk_p600_tg2": (dict(con="QPSK", Nc=600, Tg=2), dict(), K(False, False, 0, False)),
    "qpsk_c4_1344w_reg": (dict(con="QPSK", comb=4, SpF=14, reg=True), dict(near=1e-3), K(False, True, 0, False)),
    "8psk_unaligned_near_reg": (dict(con="8PSK", reg=True), dict(near=1e-3), K(False, True, 0, False)),     # 17,892-bit frames
    "8psk_unaligned_799w_noscr": (dict(con="8PSK", SpF=10), dict(scramble=False), K(False, False, 0, False)),
    "8psk_p1000_780w_near": (dict(con="8PSK", Nc=1000, SpF=10), dict(near=1e-3, two=True), K(False, True, 0, False)),
    # fallbacks to the generic kernel
    "fb_odd_tg": (dict(comb=4, Tg=511), dict(near=1e-3), GEN_RX),
    "fb_rx_offset": (dict(comb=4, reg=True), dict(near=1e-3, rx_offset=True), GEN_RX),
    "fb_nc2048": (dict(Nc=2048), dict(near=1e-3), GEN_RX),
    "fb_c4_spf27": (dict(comb=4, SpF=27, frames=1), dict(near=1e-3), GEN_RX),        # one step past the shared-memory limit
}
FALLBACKS = [k for k in RX_CASES if k.startswith("fb_")]


@pytest.mark.parametrize("case", list(RX_CASES))
def test_rx_matrix_against_oracle(G, monkeypatch, case):
    import torch
    link, opt, want = RX_CASES[case]
    p = _link(**link)
    scramble = opt.get("scramble", True)
    near_eps = opt.get("near", 0.0)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p, scramble)
    B = 3
    bits, rx = _streams(p, B, seed=sum(map(ord, case)), scramble=scramble)
    refs = [OC.rx_chain_task5(p, rx[b].astype(np.complex128), bits[b], descramble=scramble, fast=True) for b in range(B)]
    rx_d = ctx.cplx(rx)
    if opt.get("rx_offset"):
        buf = torch.empty(rx_d.numel() + 1, dtype=rx_d.dtype, device=ctx.device)
        buf[1:] = rx_d.reshape(-1)
        rx_d = buf[1:]
        assert rx_d.data_ptr() % 16 == 8
    tx_d = ctx.bits(bits.ravel())
    if opt.get("tx_offset"):
        buf = torch.zeros(tx_d.numel() + 1, dtype=tx_d.dtype, device=ctx.device)
        buf[1:] = tx_d
        tx_d = buf[1:]
        assert tx_d.data_ptr() % 16 == 4
    if opt.get("two"):
        monkeypatch.setenv("OFDM_B200_NO_SLIM", "1")
    res, kernels = _witness(lambda: ctx.rx_chain_t5(lp, rx_d, B, tx_bits_dev=tx_d, near_eps=near_eps, want_err_per_stream=True))
    _expect(kernels, want, case)
    _check_rx(ctx, p, res, refs, bits, near_eps, scramble)
    _W.ran.add(case)


# ------------------------------------------------------------------------------------------------------------- batch geometry
@pytest.fixture(scope="module")
def batch_streams(G):
    """3 x SMs + 1 comb-4 streams (device TX chain, Philox channel at 14 dB) and their host copies."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    p = _link(comb=4, reg=True)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    Bmax = 3 * sms + 1
    g = torch.Generator(device=ctx.device)
    g.manual_seed(21)
    bd = torch.randint(-2**31, 2**31 - 1, (Bmax * p.stream_bits // 32,), dtype=torch.int32, device=ctx.device, generator=g)
    tx, ps = ctx.tx_chain(lp, bd, Bmax, want_power=True)
    rx = ctx.channel_t5(tx, snr_db=14.0, h_dev=ctx.cplx(O.get_MP_channel_resp(TAPS5, p.Nfft)[0]), seed=8, power_sum=ps)
    ctx.sync()
    return dict(sms=sms, p=p, lp=lp, Bmax=Bmax, bits_d=bd, rx_d=rx, bits=ctx.host_bits(bd, Bmax * p.stream_bits).reshape(Bmax, -1),
                rx=rx.cpu().numpy().reshape(Bmax, -1))


@pytest.mark.parametrize("variant", ["three", "two"])
def test_batch_geometry_around_the_persistent_grid(G, monkeypatch, batch_streams, variant):
    """B = 1 and grid - 1, grid, grid + 1 (grid = 3 x SMs for the three-CTA kernel, 2 x SMs for the two-CTA one): every stream
    against the generic kernel, the first, the last, streams grid - 1 and grid and four random ones against the oracle."""
    import torch
    bs = batch_streams
    p, lp = bs["p"], bs["lp"]
    ctx = G.default_context("f32")
    grid = (3 if variant == "three" else 2) * bs["sms"]
    words = p.stream_bits // 32
    rng = np.random.default_rng(grid)
    for B in (1, grid - 1, grid, grid + 1):
        rx_d = bs["rx_d"][:B]
        tx_d = bs["bits_d"][:B * words]
        if variant == "two":
            monkeypatch.setenv("OFDM_B200_NO_SLIM", "1")
        fast, kernels = _witness(lambda: ctx.rx_chain_t5(lp, rx_d, B, tx_bits_dev=tx_d, near_eps=1e-3, want_err_per_stream=True))
        _expect(kernels, K(True, True, 0x1111, variant == "three"), f"batch_{variant}_{B}")
        monkeypatch.delenv("OFDM_B200_NO_SLIM", raising=False)
        monkeypatch.setenv("OFDM_B200_NO_FAST", "1")
        gen, kernels = _witness(lambda: ctx.rx_chain_t5(lp, rx_d, B, tx_bits_dev=tx_d, near_eps=1e-3, want_err_per_stream=True))
        _expect(kernels, GEN_RX, f"batch_generic_{B}")
        monkeypatch.delenv("OFDM_B200_NO_FAST")
        cf, cg = fast["counts"].cpu().numpy(), gen["counts"].cpu().numpy()
        Hf, Hg = fast["H"].cpu().numpy(), gen["H"].cpu().numpy()
        assert np.all(np.linalg.norm(Hf - Hg, axis=1) < 2e-5 * np.linalg.norm(Hg, axis=1))
        got = ctx.host_bits(fast["bits"], B * p.stream_bits).reshape(B, -1)
        got_g = ctx.host_bits(gen["bits"], B * p.stream_bits).reshape(B, -1)
        assert int(np.sum(got != got_g)) <= 3 * p.bps * int(cf[2] + cg[2])
        per_stream = (got != bs["bits"][:B]).sum(axis=1)
        assert np.array_equal(fast["err_per_stream"].cpu().numpy(), per_stream)
        assert cf[0] == per_stream.sum() and cf[1] == cg[1] == B * p.stream_bits
        sample = {0, B - 1, grid - 1, grid} | set(rng.integers(0, B, 4).tolist())
        for b in sorted(s for s in sample if s < B):
            ref = OC.rx_chain_task5(p, bs["rx"][b].astype(np.complex128), bs["bits"][b], fast=True)
            assert rel_err(Hf[b], ref["H"]) < 2e-5, (B, b)
            _check_stream(p, got[b], ref)


# ------------------------------------------------------------------------------------------------------------- near counter, host entry
def test_host_entry_returns_the_near_boundary_count(G):
    """ofdm_rx_chain_t5_host_eps (CP stripped on the host, Tg = 0 on the device, chunks of 4) returns the device entry's three
    counters, the near-boundary count included, and its decided bits and channel estimates."""
    import torch
    p = _link(comb=4, reg=True)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    B = 10
    bits, rx = _streams(p, B, seed=10)
    rx_d, bd = ctx.cplx(rx), ctx.bits(bits.ravel())
    dev = ctx.rx_chain_t5(lp, rx_d, B, tx_bits_dev=bd, near_eps=1e-3)
    ctx.sync()
    rx_h = rx_d.cpu().pin_memory()
    tb_h = bd.cpu().pin_memory()
    ob_h = torch.zeros_like(tb_h).pin_memory()
    H_h = torch.zeros((B, p.N_carrier), dtype=torch.complex64).pin_memory()
    counts = ctx.rx_chain_t5_host(lp, rx_h, B, tb_h, ob_h, H_h, chunk=4, near_eps=1e-3)
    dc = dev["counts"].cpu().numpy()
    assert dc[2] > 0 and np.array_equal(counts, dc)
    assert torch.equal(ob_h, dev["bits"].cpu()) and torch.equal(torch.view_as_real(H_h), torch.view_as_real(dev["H"].cpu()))


# ------------------------------------------------------------------------------------------------------------- optional outputs
@pytest.mark.parametrize("comb", [4, 7])
@pytest.mark.parametrize("variant", ["three", "two"])
def test_optional_outputs_and_buffer_hygiene(G, monkeypatch, comb, variant):
    """Each of out_bits, H, err_per_stream and tx_bits omitted in turn; outputs pre-filled with garbage (0xA5A5A5A5, NaN, -1)
    come back exactly as a call on zeroed buffers writes them; the counters accumulate over calls."""
    import torch
    p = _link(comb=comb, reg=True)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    B = 4
    bits, rx = _streams(p, B, seed=comb)
    rx_d, tx_d = ctx.cplx(rx), ctx.bits(bits.ravel())
    words = (B * p.stream_bits + 31) // 32
    if variant == "two":
        monkeypatch.setenv("OFDM_B200_NO_SLIM", "1")
    want = K(True, True, 0x1111 if comb == 4 else 0, variant == "three")

    def call(tx=True, ob=True, H=True, eps=True, counts=None):
        ob_t = torch.full((words,), -0x5A5A5A5B, dtype=torch.int32, device=ctx.device) if ob else None    # 0xA5A5A5A5
        H_t = torch.full((B, p.N_carrier), complex(np.nan, np.nan), dtype=torch.complex64, device=ctx.device) if H else None
        e_t = torch.full((B,), -1, dtype=torch.int32, device=ctx.device) if eps else None
        c_t = torch.zeros(3, dtype=torch.int64, device=ctx.device) if counts is None else counts
        ctx._chk(ctx.lib.ofdm_rx_chain_t5(ctx.h, C.byref(lp), ctx.p(rx_d), B, ctx.p(tx_d if tx else None), ctx.p(ob_t), ctx.p(H_t),
                                          ctx.p(c_t), ctx.p(e_t), 1e-3))
        ctx.sync()
        return ob_t, H_t, c_t, e_t

    ref = ctx.rx_chain_t5(lp, rx_d, B, tx_bits_dev=tx_d, near_eps=1e-3, want_err_per_stream=True)    # zero-filled buffers
    ctx.sync()
    r_ob, r_H, r_c, r_e = ref["bits"], torch.view_as_real(ref["H"]), ref["counts"], ref["err_per_stream"]
    assert int(r_c[0]) > 0 and int(r_c[2]) > 0
    (ob, H, c, e), kernels = _witness(call)
    _expect(kernels, want, f"hygiene_c{comb}_{variant}")
    assert torch.equal(ob, r_ob) and torch.equal(torch.view_as_real(H), r_H) and torch.equal(c, r_c) and torch.equal(e, r_e)
    ob, H, c, e = call(ob=False)
    assert torch.equal(torch.view_as_real(H), r_H) and torch.equal(c, r_c) and torch.equal(e, r_e)
    ob, H, c, e = call(H=False)
    assert torch.equal(ob, r_ob) and torch.equal(c, r_c) and torch.equal(e, r_e)
    ob, H, c, e = call(eps=False)
    assert torch.equal(ob, r_ob) and torch.equal(torch.view_as_real(H), r_H) and torch.equal(c, r_c)
    ob, H, c, e = call(tx=False)
    assert torch.equal(ob, r_ob) and torch.equal(torch.view_as_real(H), r_H) and int(e.abs().sum()) == 0
    assert int(c[0]) == 0 and int(c[1]) == B * p.stream_bits and int(c[2]) == int(r_c[2])
    acc = torch.zeros(3, dtype=torch.int64, device=ctx.device)
    call(counts=acc)
    call(counts=acc)
    assert torch.equal(acc, 2 * r_c)


# ------------------------------------------------------------------------------------------------------------- TX matrix
TX_CASES = {
    "16qam_c8_25088b_reg": (dict(comb=8, reg=True), True),                   # frames > 24,576 bits: words fetched on the spot
    "16qam_c4_79872b_tg0": (dict(comb=4, SpF=26, frames=1, Tg=0), True),     # two more scrambler doublings than 24,576 bits need
    "16qam_p600_noscr": (dict(Nc=600), False),
    "bpsk_p600_tg0_reg": (dict(con="BPSK", Nc=600, Tg=0, reg=True), True),
    "bpsk_noscr_tg2": (dict(con="BPSK", Tg=2), False),
    "qpsk_c4_30720b_reg": (dict(con="QPSK", comb=4, SpF=20, reg=True), True),
    "qpsk_p1000_noscr_tg0": (dict(con="QPSK", Nc=1000, Tg=0), False),
    "8psk_25560b_reg": (dict(con="8PSK", SpF=10, reg=True), True),           # unaligned frames through sm_get32
    "8psk_p600_noscr_tg0": (dict(con="8PSK", Nc=600, Tg=0), False),
}


@pytest.mark.parametrize("case", list(TX_CASES))
def test_tx4096_matrix_against_oracle(G, case):
    link, scramble = TX_CASES[case]
    p = _link(**link)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p, scramble)
    rng = np.random.default_rng(sum(map(ord, case)))
    B = 3
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    (tx, ps), kernels = _witness(lambda: ctx.tx_chain(lp, ctx.bits(bits.ravel()), B, want_power=True))
    _expect(kernels, TX4096, f"tx_{case}")
    tx_h = tx.cpu().numpy().reshape(B, -1)
    ps = ps.cpu().numpy()
    for b in range(B):
        ref, _, _ = OC.tx_chain(p, bits[b], scramble=scramble, fast=True)
        assert rel_err(tx_h[b], ref) < 2e-6, b
        assert abs(ps[b] / np.sum(np.abs(ref) ** 2) - 1) < 1e-5, b


# ------------------------------------------------------------------------------------------------------------- per-symbol pilots
@pytest.mark.parametrize("entry", ["tx4096", "tx1024", "generic_f64"])
def test_per_symbol_pilots_tx(G, entry):
    """Np x S pilot values with distinct columns and a random register: symbol s carries column s."""
    rng = np.random.default_rng(77)
    if entry == "tx4096":
        p, prec, want, tol = _link(comb=4, reg=True), "f32", TX4096, 2e-6
    elif entry == "tx1024":
        p, prec, tol = OC.params_task4(), "f32", 2e-6
        want = ("tx1024_kernel", ())
    else:
        p, prec, want, tol = _link(Nfft=2048, Nc=800, Tg=256, SpF=5, frames=2), "f64", ("tx_chain_kernel", ("double",)), 1e-12
    p.Register = rng.integers(0, 2, 15).astype(np.uint8)
    p.Register[12:14] = 1
    _random_pilots(p, rng)
    ctx = G.default_context(prec)
    lp = _lp(ctx, p)
    B = 3
    bits = rng.integers(0, 2, (B, p.stream_bits)).astype(np.uint8)
    tx, kernels = _witness(lambda: ctx.tx_chain(lp, ctx.bits(bits.ravel()), B))
    _expect(kernels, want, f"pilots_{entry}")
    tx_h = tx.cpu().numpy().reshape(B, -1)
    for b in range(B):
        ref, _, _ = OC.tx_chain(p, bits[b], fast=True)
        assert rel_err(tx_h[b], ref) < tol, b


@pytest.mark.parametrize("path", ["fast", "generic"])
def test_per_symbol_pilots_rx_t5(G, monkeypatch, path):
    """The M1 receiver estimates from symbol 0 (`LS_CE.m:27-28`): it must divide by column 0 of the pilot matrix."""
    rng = np.random.default_rng(78)
    p = _random_pilots(_link(comb=4, reg=True), rng)
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    B = 3
    bits, rx = _streams(p, B, seed=78)
    refs = [OC.rx_chain_task5(p, rx[b].astype(np.complex128), bits[b], fast=True) for b in range(B)]
    if path == "generic":
        monkeypatch.setenv("OFDM_B200_NO_FAST", "1")
    rx_d, bd = ctx.cplx(rx), ctx.bits(bits.ravel())
    res, kernels = _witness(lambda: ctx.rx_chain_t5(lp, rx_d, B, tx_bits_dev=bd, near_eps=1e-3, want_err_per_stream=True))
    _expect(kernels, K(True, True, 0x1111, True) if path == "fast" else GEN_RX, f"pilots_t5_{path}")
    _check_rx(ctx, p, res, refs, bits, 1e-3)


@pytest.mark.parametrize("path", ["split", "fused"])
def test_per_symbol_pilots_rx_t4(G, monkeypatch, path):
    """fine_sync and estimate_channel of the Task-4 receiver use every pilot column (`fine_sync.m:26-27`, `estimate_channel.m:6`):
    the split chain (from 512 streams on) and the fused kernel against the oracle, with the tolerances of test_gpu_chain.py; the
    phase estimate within FP32 rounding of the interval that the signs of exact zeros leave open (_t4_phase_bounds)."""
    TAPS4 = [[0, 1], [4, .6], [10, .3]]
    rng = np.random.default_rng(79)
    p = OC.params_task4()
    p.Register = REG.copy()
    _random_pilots(p, rng, 4.0 / 3.0, jitter=0.0)     # equal magnitudes: remove_IFO looks for the strongest bins
    ctx = G.default_context("f32")
    lp = _lp(ctx, p)
    cases = [(37, 7.24), (900, 0.24), (150, 12.4), (0, 0.0), (611, 3.3), (1152, 30.4), (1, 0.49), (77, 21.7)]
    n = len(cases)
    bits = rng.integers(0, 2, (n, p.stream_bits)).astype(np.uint8)
    rxs, refs = [], []
    for b, (sto, cfo) in enumerate(cases):
        tx, _, _ = OC.tx_chain(p, bits[b], fast=True)
        rx = OC.impair_task4(p, tx, SNR_dB=28, Time_Delay=sto, Freq_Shift=cfo, taps=TAPS4, rng=rng).astype(np.complex64)
        rxs.append(rx)
        refs.append(OC.rx_chain_task4(p, rx.astype(np.complex128), bits[b]))
    reps = 65 if path == "split" else 1                     # >= 512 streams select the split chain
    B = n * reps
    rx_d = ctx.cplx(np.tile(np.stack(rxs), (reps, 1)))
    bd = ctx.bits(np.tile(bits, (reps, 1)).ravel())
    if path == "fused":
        monkeypatch.setenv("OFDM_B200_T4_FUSED", "1")
    out, kernels = _witness(lambda: ctx.rx_chain_t4_fused(lp, rx_d, tx_bits_dev=bd, near_eps=1e-3, want_H=True))
    if kernels is not None:
        names = {k[0] for k in kernels}
        assert ("t4_post_kernel" in names) == (path == "split") and ("rx_t4_fast_kernel" in names) == (path == "fused"), names
    got = ctx.host_bits(out["bits"], B * p.stream_bits).reshape(B, -1)
    tg, ifo = out["TgPosition"].cpu().numpy(), out["IFO"].cpu().numpy()
    fo, tau, ph = out["FreqOffset"].cpu().numpy(), out["tau"].cpu().numpy(), out["phase_shift"].cpu().numpy()
    H = out["H"].cpu().numpy()

    def close(a, r, tol):      # NaN is a legitimate result of the reference algorithm (mean of an empty selection)
        return (np.isnan(a) and np.isnan(r)) or abs(a - r) < tol
    mism, n_finite = 0, 0
    for b in range(n):
        assert tg[b] == refs[b]["TgPosition"] and ifo[b] == refs[b]["IFO"], b
        assert close(fo[b], refs[b]["FreqOffset"], 2e-5) and close(tau[b], refs[b]["tau"], 2e-5), b
        if np.isnan(refs[b]["phase_shift"]):
            assert np.isnan(ph[b]), b
        else:
            lo, hi = _t4_phase_bounds(p, rxs[b], refs[b])
            assert lo - 2e-3 < ph[b] < hi + 2e-3, (b, lo, ph[b], hi)
        Href = refs[b]["H"][:p.N_carrier]
        if np.all(np.isfinite(Href)):
            dphi = ph[b] - refs[b]["phase_shift"]
            assert np.linalg.norm(H[b] * np.exp(-1j * dphi) - Href) / np.linalg.norm(Href) < 1e-3, b
            mism += int(np.sum(got[b] != refs[b]["bits"]))
            n_finite += 1
    assert n_finite >= 4
    counts = out["counts"].cpu().numpy()
    assert counts[1] == B * p.stream_bits and counts[0] == int(np.sum(got != np.tile(bits, (reps, 1))))
    assert mism * reps <= 3 * p.bps * int(counts[2])


# ------------------------------------------------------------------------------------------------------------- coverage
def test_witness_covered_every_instantiation():
    """The cases above together launched all 14 rx4096_kernel instantiations, tx4096_kernel, and the generic receiver for each
    fallback (odd guard, misaligned rx, N_carrier > 1024, shared memory over the limit)."""
    if _W.available is False:
        pytest.skip("the profiler recorded no CUDA activity (no CUPTI): kernel identities are not observable here")
    if _W.available is None or set(RX_CASES) - _W.ran:
        pytest.skip("kernel coverage needs every RX case of this module in the same session")
    want = {K(True, n, m, s) for n in (False, True) for m in (0x1111, 0x0101, 0) for s in (False, True)}
    want |= {K(False, n, 0, False) for n in (False, True)}
    seen = {k for k in _W.seen if k[0] == "rx4096_kernel"}
    print("rx4096_kernel instantiations observed:", sorted(k[1] for k in seen))
    print("generic receiver observed for:", sorted(_W.seen.get(GEN_RX, ())))
    assert len(want) == 14 and want <= seen, sorted(want - seen)
    assert TX4096 in _W.seen
    assert set(FALLBACKS) <= _W.seen.get(GEN_RX, set())
