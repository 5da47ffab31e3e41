"""ofdm_sweep_mse (the channel-estimation MSE-vs-SNR loop of `Task 5/Main_model_Task_5.m:303-346`) on the GPU: bit-identical
to the same streams pushed through the exported calls one by one, independent of tile size and rank count, close to the
float64 oracle, on the analytic noise budget, and the same through the MEX gateway."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O

pytestmark = pytest.mark.gpu

TAPS = [[0, 1], [4, .8], [10, .6], [15, .4], [21, .2], [25, .1]]      # `Main_model_Task_5.m:112-119`
NFFT, NC, TG, S = 4096, 1024, 512, 14


def _ctx(prec="f32"):
    import ofdm_b200 as G
    return G.default_context(prec)


def _layout(comb):
    pc = np.arange(1, NC + 1)[::comb]
    dc = np.setdiff1d(np.arange(1, NC + 1), pc)
    amp = 4.0 / 3.0 * np.max(np.abs(O.constellation_func("16QAM")[0]))
    pv = np.tile(np.conj(np.full(pc.size, amp * np.exp(1j * 0)))[:, None], (1, S))
    return pc, dc, pv, amp


def _link(ctx, comb):
    pc, dc, pv, _ = _layout(comb)
    return ctx.link_params(NFFT, TG, NC, S, 7, "16QAM", dc, pc, pv, scramble=False)


def _ldict(comb):
    return -(-NC // comb)


def _composed(ctx, lp, snrs, spp, seed, tie_eps, keep_rx=None):
    """The sweep written out as exported calls: TX of stream g, channel_t5 -> demodulate -> ls_ce, then ifft -> mmse_ce ->
    pilot_ls -> mp -> omp -> mse x 4.  Returns (per_stream [n_snr, 4, spp], counts [n_snr, 2], rx of point i if asked)."""
    pc, pv = lp.pilotCarriers, lp.pilotValues
    K = len(TAPS)
    Ldict = _ldict(int(pc[1] - pc[0]))
    h, Htrue = ctx.mp_channel_resp(TAPS, NFFT)
    h_dev = ctx.cplx(h)
    per = np.zeros((len(snrs), 4, spp))
    counts = np.zeros((len(snrs), 2), dtype=np.int64)
    rx_out = {}
    for i, snr in enumerate(snrs):
        g0 = i * spp
        if lp.Nd == 0:                                   # pilots only: one TX stream for every g, its power measured by the channel
            tx1 = ctx.modulate(ctx.map_carriers(None, 1, S, NFFT, [], pc, pv), TG)
            tx, psum = tx1.expand(spp, -1, -1).contiguous(), None
        else:                                            # what ofdm_sweep_ber transmits for stream g
            words = lp.stream_bits // 32
            bits = torch.empty(spp * words, dtype=torch.int32, device=ctx.device)
            ctx._chk(ctx.lib.ofdm_payload_bits(ctx.h, ctx.p(bits), spp, words, seed, g0))
            tx, psum = ctx.tx_chain(lp, bits, spp, want_power=True)
        rx = ctx.channel_t5(tx, snr_db=float(snr), h_dev=h_dev, seed=seed, first_stream_id=g0, power_sum=psum)
        if keep_rx is not None and i in keep_rx:
            rx_out[i] = rx.cpu().numpy()
        Y = ctx.demodulate(rx, NFFT, TG)
        H_ls = ctx.ls_ce(Y, pv, pc, NC)
        H_mm = ctx.mmse_ce(Y, pv, pc, NC, ctx.fft(H_ls, inverse=True), float(snr))
        y = ctx.pilot_ls(Y, pv, pc)
        H_mp = ctx.mp(y, NFFT, K, Ldict=Ldict, pilot_loc=pc)[0]
        H_omp, _, _, _, near = ctx.omp(y, NFFT, K, Ldict=Ldict, pilot_loc=pc, tie_eps=tie_eps)
        ref = Htrue[None].expand(spp, -1).contiguous()
        for e, H in enumerate((H_ls, H_mm, H_mp, H_omp)):
            per[i, e] = ctx.mse(ref, H, NC).cpu().numpy()
        counts[i] = (spp, int((near != 0).sum().item()))
    return per, counts, rx_out


@pytest.mark.parametrize("prec,comb", [("f32", 1), ("f32", 4), ("f64", 1)])
def test_sweep_equals_composed_calls(prec, comb):
    from ofdm_b200 import sweep
    ctx = _ctx(prec)
    lp = _link(ctx, comb)
    assert lp.Nd == (0 if comb == 1 else 768)
    snrs, spp, seed, eps = [0.0, 12.5, 30.0], 300, 5, 1e-3
    mean, per, counts = sweep.mse_sweep(ctx, lp, snrs, spp, TAPS, seed=seed, tile=128, tie_eps=eps)       # ragged tiles
    want, wcounts, _ = _composed(ctx, lp, snrs, spp, seed, eps)
    assert np.array_equal(per, want)
    assert np.array_equal(counts, wcounts) and np.all(counts[:, 0] == spp)
    assert np.array_equal(mean, want.mean(axis=2))
    assert np.all(np.isfinite(per)) and np.all(per > 0)


def test_tile_and_rank_count_do_not_change_the_result():
    from ofdm_b200 import sweep
    ctx = _ctx("f32")
    lp = _link(ctx, 1)
    snrs, spp, seed = [0.0, 12.5, 30.0], 300, 9
    _, per1, cnt1 = sweep.mse_sweep(ctx, lp, snrs, spp, TAPS, seed=seed, tie_eps=1e-3)
    _, per2, cnt2 = sweep.mse_sweep(ctx, lp, snrs, spp, TAPS, seed=seed, tile=1000, tie_eps=1e-3)
    per3 = torch.zeros((len(snrs), 4, spp), dtype=torch.float64, device=ctx.device)
    cnt3 = torch.zeros((len(snrs), 2), dtype=torch.int64, device=ctx.device)
    for r in range(3):                                   # three ranks' calls into one buffer
        sweep.mse_sweep_local(ctx, lp, snrs, spp, TAPS, seed=seed, rank=r, world=3, tile=77, tie_eps=1e-3, per_stream=per3, counts=cnt3)
    ctx.sync()
    for per, cnt in ((per2, cnt2), (per3.cpu().numpy(), cnt3.cpu().numpy())):
        assert np.array_equal(per, per1) and np.array_equal(cnt, cnt1)


@pytest.mark.parametrize("prec,tol", [("f64", 1e-8), ("f32", 1e-3)])
def test_against_oracle(prec, tol):
    """The composed rx of 8 streams per point through the oracle's LS_CE / MMSE_CE / MP / OMP and MSE."""
    from ofdm_b200 import sweep
    ctx = _ctx(prec)
    lp = _link(ctx, 1)
    pc, _, pv, _ = _layout(1)
    snrs, spp, seed, eps = [5.0, 20.0], 8, 3, 1e-3
    _, per, counts = sweep.mse_sweep(ctx, lp, snrs, spp, TAPS, seed=seed, tie_eps=eps)
    _, _, rx = _composed(ctx, lp, snrs, spp, seed, eps, keep_rx=(0, 1))
    _, Hf = O.get_MP_channel_resp(TAPS, NFFT)
    Hu = np.asarray(Hf).ravel()[:NC]
    A = O.sensing_matrix_dft(pc, NFFT, _ldict(1))
    mse = lambda H: float(np.sum(np.abs(Hu - np.asarray(H).ravel()[:NC]) ** 2) / NC)   # noqa: E731, `:195-205`
    for i, snr in enumerate(snrs):
        outside = 0
        for j in range(spp):
            Y = O.OFDM_demodulator(rx[i][j].ravel().astype(np.complex128).reshape((NFFT + TG, S), order="F"), TG)
            H_ls = O.LS_CE(Y, pv, pc, NC)
            H_mm = O.MMSE_CE(Y, pv, pc, NFFT, NC, np.fft.ifft(H_ls), snr)
            y = Y[pc - 1, 0] / pv[:, 0]
            H_mp, _ = O.MP_estimate(y, A, NFFT, len(TAPS))
            H_omp, _, _ = O.OMP_estimate(y, A, NFFT, len(TAPS), snr)
            ref = np.array([mse(H_ls), mse(H_mm), mse(H_mp), mse(H_omp)])
            outside += int(np.any(np.abs(per[i, :, j] - ref) > tol * ref))
        assert outside <= counts[i, 1], (snr, outside, counts[i])


def test_noise_budget_and_the_scripts_conclusion():
    """Comb 1: every carrier of N_carrier is a pilot, so H_LS = Y/a and its MSE is the noise power per bin over a^2.  The noise
    is white before the FIR, so E|N_k|^2 = Nfft NP sum_tau r_h(tau) (1 - |tau|/Nfft) exp(-2j pi k tau / Nfft)."""
    from ofdm_b200 import sweep
    ctx = _ctx("f32")
    lp = _link(ctx, 1)
    pc, _, pv, amp = _layout(1)
    snrs = [0.0, 10.0, 20.0, 30.0]
    mean, _, counts = sweep.mse_sweep(ctx, lp, snrs, 2048, TAPS, seed=11)
    assert np.all(counts[:, 0] == 2048)
    grid = np.zeros((NFFT, S), dtype=np.complex128)
    grid[pc - 1, :] = pv
    P = np.mean(np.abs(O.OFDM_modulator(grid, TG)) ** 2)          # power of the whole stream, `Noise.m:3`
    h, _ = O.get_MP_channel_resp(TAPS, NFFT)
    h = np.asarray(h, dtype=complex).ravel()
    D = h.size
    taus = np.arange(-(D - 1), D)
    r_h = np.array([sum(h[m + t] * np.conj(h[m]) for m in range(D) if 0 <= m + t < D) for t in taus])
    k = np.arange(NC)[:, None]
    Sk = np.real(np.sum(r_h[None, :] * (1 - np.abs(taus[None, :]) / NFFT) * np.exp(-2j * np.pi * k * taus[None, :] / NFFT), axis=1))
    for i, snr in enumerate(snrs):
        NP = P / 10 ** (snr / 10)
        want = np.mean(NFFT * NP * Sk) / amp ** 2
        assert abs(mean[i, 0] / want - 1) < 0.02, (snr, mean[i, 0], want)
    assert np.all(np.diff(mean[:, 0]) < 0)                      # LS MSE falls with SNR
    # the script's conclusion (asserted for one stream at 20 dB in test_gpu_task5_main.py): the sparse estimate beats LS.
    # At 30 dB it does not: OMP_estimate's stopping rule leaves a floor of ~2.9e-3 (the float64 oracle gives the same on its
    # own noise draws), while LS is at ~6.8e-4.
    assert np.all(mean[:3, 3] < mean[:3, 0])
    assert 2e-3 < mean[3, 3] < 4e-3 and mean[3, 3] > mean[3, 0]


def test_mex_gateway_equals_python():
    import os
    import subprocess
    from ofdm_b200 import sweep
    from test_gpu_mex import Mex
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["make", "-C", os.path.join(root, "mex")], check=True, capture_output=True)
    mex = Mex("interleaved")
    ctx = _ctx("f32")
    reg = O.DEFAULT_REGISTER.astype(float)
    try:
        for comb in (1, 4):
            pc, dc, pv, _ = _layout(comb)
            lp = _link(ctx, comb)
            snrs, spp = [5.0, 15.0], 6
            args = [float(NFFT), float(TG), float(NC), float(S), 7.0, "16QAM", dc.astype(float), pc.astype(float), pv[:, :1], reg]
            got_m, got_p, got_c = mex.call("sweep_mse", *args, np.asarray(snrs), float(spp), np.asarray(TAPS, dtype=float), 3.0, 1e-3, nout=3)
            mean, per, counts = sweep.mse_sweep(ctx, lp, snrs, spp, TAPS, seed=3, tie_eps=1e-3)
            assert got_p.shape == (spp, 4 * len(snrs))
            assert np.array_equal(got_p.reshape(spp, 4, len(snrs), order="F").transpose(2, 1, 0), per)
            assert np.array_equal(got_c.astype(np.int64), counts)
            assert np.allclose(got_m, mean, rtol=1e-13, atol=0)          # the gateway sums the streams in order
    finally:
        mex.lib.ofdm_mex_shim_exit()


def test_rejections():
    from ofdm_b200 import _cabi
    ctx = _ctx("f32")
    lp = _link(ctx, 1)
    snr = np.array([10.0])
    per = torch.zeros((1, 4, 4), dtype=torch.float64, device=ctx.device)
    cnt = torch.zeros((1, 2), dtype=torch.int64, device=ctx.device)

    def params(taps=TAPS, chain=0):
        sp = _cabi.SweepParams()
        sp.chain, sp.n_snr, sp.snr_db_host = chain, 1, snr.ctypes.data_as(_cabi.pdbl)
        sp.streams_per_point, sp.rank, sp.world, sp.seed = 4, 0, 1, 1
        t = np.ascontiguousarray(np.asarray(taps, dtype=np.float64).reshape(-1, 2))
        sp._t = t
        sp.taps_host, sp.n_taps = t.ctypes.data_as(_cabi.pdbl), t.shape[0]
        return sp

    call = lambda l, s, Ld=1024, m=per, c=cnt: ctx.lib.ofdm_sweep_mse(ctx.h, C.byref(l) if l is not None else None,   # noqa: E731
                                                                        C.byref(s) if s is not None else None, Ld, ctx.p(m), ctx.p(c))
    assert call(lp, params()) == 0
    ctx.sync()
    assert call(None, params()) == -1 and call(lp, None) == -1
    assert call(lp, params(), m=None) == -1 and call(lp, params(), c=None) == -1
    zero = params()
    zero.n_taps = 0
    assert call(lp, zero) == -1                                               # no channel
    assert call(lp, params(taps=[[d, 0.5] for d in range(33)])) == -1         # K > 32
    assert call(lp, params(), Ld=1023) == -1                                  # Ldict < Np
    assert call(lp, params(chain=1)) == -1                                    # chain != TASK5
    pc, dc, pv, _ = _layout(1)
    odd = ctx.link_params(NFFT, TG, 1000, S, 7, "16QAM", dc, pc[:1000], pv[:1000], scramble=False)
    assert call(odd, params(), Ld=1000) == -1                                 # N_carrier not a power of two
    assert "power of two" in ctx.lib.ofdm_last_error(ctx.h).decode()
