"""ofdm_sweep_part2 (the pilot-density study of `Task 5/Task5_part2.m:46-321`) on the GPU: bit-identical to the composed
exported calls of part2.run_point / part2.sweep, independent of tile size and rank count, within the library's own
near-boundary count of the float64 oracle, a sane experiment, the same through the MEX gateway, and every argument check."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import chains as OC

pytestmark = pytest.mark.gpu

NFFT, NC, S, SNR, FS = 4096, 1024, 14, 20.0, 4e7
ALL_BITS = np.random.default_rng(2024).integers(0, 2, S * NC * 4).astype(np.uint8)      # longer than any point's stream


def _ctx(prec="f32"):
    import ofdm_b200 as G
    return G.default_context(prec)


def _omp_ties(ctx, part2, Y, pc, n_paths, Ldict, amp, tie_eps):
    pv = part2.pilot_values(len(pc), S, amp)
    y = ctx.pilot_ls(Y, pv, pc)
    near = ctx.omp(y, NFFT, n_paths, Ldict=Ldict, pilot_loc=pc, tie_eps=tie_eps)[4]
    return int((near != 0).sum().item())


@pytest.mark.parametrize("profile", ["EPA", "ETU"])
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_sweep_lib_equals_composed_calls(prec, profile):
    from ofdm_b200 import link as G
    from ofdm_b200 import part2
    ctx = _ctx(prec)
    runs, seed, eps = 7, 13, 1e-3
    amp = 2.0 * float(np.max(np.abs(G.constellation_func("16QAM")[0])))
    n_paths, _, _ = ctx.tdl_info(profile, FS)
    mask = np.sort(np.random.default_rng(5).permutation(NC)[:64]) + 1
    kw = dict(profile=profile, fs_hz=FS, snr_db=SNR, seed=seed)
    # comb 5 (Nd 819) sends a stream of S * Nd * bps bits that ends inside a 32-bit word; the others end on a word boundary
    for combs, reg, masks in (([4, 5, 37, 256], True, None), ([0], False, [mask])):
        NMSE, BER, per, counts, rn = part2.sweep_lib(ctx, combs, runs, ALL_BITS, tile=3, reg_pilot=reg, random_masks=masks,  # ragged tiles
                                                     tie_eps=eps, **kw)
        off, car, ldict = part2.lib_layout(combs, reg_pilot=reg, random_masks=masks)
        for k in range(len(combs)):
            pc, dc = part2.layout(NC, pilotCarriers=car[off[k]:off[k + 1]])
            n = S * dc.size * 4
            nmse, errs, nbits, ex = part2.run_point(ctx, pc, dc, ALL_BITS[:n], runs, point_id=k, first_run=0, Ldict=int(ldict[k]), **kw)
            assert np.array_equal(per[k].T, nmse), (combs[k], k)
            assert np.array_equal(counts[k, :, 0], errs) and np.all(counts[k, :, 1] == runs * nbits)
            assert rn[k, 0] == runs and rn[k, 1] == _omp_ties(ctx, part2, ex["Y"], pc, n_paths, int(ldict[k]), amp, eps)
        N2, B2 = part2.sweep(ctx, combs, runs, lambda n: ALL_BITS[:n], block=4, reg_pilot=reg, random_masks=masks, **kw)
        assert np.array_equal(NMSE, N2) and np.array_equal(BER, B2)
        assert np.all(np.isfinite(per)) and np.all(per > 0)


def test_tile_and_rank_count_do_not_change_the_result():
    from ofdm_b200 import part2
    ctx = _ctx("f32")
    combs, runs = [4, 37], 160
    kw = dict(profile="EVA", fs_hz=FS, snr_db=SNR, seed=21, near_eps=1e-3, tie_eps=1e-3)
    ref = part2.sweep_lib(ctx, combs, runs, ALL_BITS, **kw)
    for tile in (1, 77):
        got = part2.sweep_lib(ctx, combs, runs, ALL_BITS, tile=tile, **kw)
        assert all(np.array_equal(a, b) for a, b in zip(got, ref)), tile
    per = torch.zeros((2, 4, runs), dtype=torch.float64, device=ctx.device)
    cnt = torch.zeros((2, 4, 3), dtype=torch.int64, device=ctx.device)
    rn = torch.zeros((2, 2), dtype=torch.int64, device=ctx.device)
    for r in range(3):                                   # three ranks' calls into one buffer
        part2.sweep_lib_local(ctx, combs, runs, ALL_BITS, tile=77, rank=r, world=3, per_run=per, counts=cnt, runs=rn, **kw)
    ctx.sync()
    got = part2.reduce_part2(per, cnt, rn)
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_error_counts_against_oracle(prec):
    """One point through the oracle's `Task5_part2.m:148-304` on the library's own noisy stream and fading responses: FP64
    error counts are exact; in FP32 a decision can only flip where the symbol is near a boundary, and with no descrambler a
    flipped symbol costs at most bps bits, so the difference is bounded by bps x the library's near-boundary count."""
    from ofdm_b200 import part2
    ctx = _ctx(prec)
    comb, runs, seed, k, near_eps = 8, 4, 17, 0, 1e-3
    p = OC.params_part2(comb=comb)
    bits = ALL_BITS[:p.stream_bits]
    Ldict = -(-NFFT // comb)
    _, _, per, counts, _ = part2.sweep_lib(ctx, [comb], runs, ALL_BITS, profile="EPA", fs_hz=FS, snr_db=SNR, seed=seed, near_eps=near_eps)
    lp = ctx.link_params(NFFT, NFFT // 8, NC, S, 7, "16QAM", p.dataCarriers, p.pilotCarriers, p.pilotValues, scramble=False)
    tx = ctx.tx_chain(lp, ctx.bits(bits), 1).reshape(1, -1)
    txn = ctx.add_noise(tx, SNR, seed=seed, first_stream_id=k)[0][0].cpu().numpy().astype(np.complex128)
    h = ctx.tdl_channel("EPA", FS, runs, seed=seed, first_stream_id=k * 1_000_003).cpu().numpy().astype(np.complex128)
    ref_err, ref_nmse = np.zeros(4, dtype=np.int64), np.zeros((4, runs))
    for r in range(runs):
        rn, re_, _ = OC.part2_run(p, txn, h[r], bits, len(OC.TDL_PROFILES["EPA"][0]), SNR, Ldict)
        ref_err += re_
        ref_nmse[:, r] = rn
    if prec == "f64":
        assert np.allclose(per[0], ref_nmse, rtol=1e-6, atol=0)
        assert np.array_equal(counts[0, :, 0], ref_err)
    else:
        assert np.all(np.abs(counts[0, :, 0] - ref_err) <= 4 * counts[0, :, 2]), (counts[0], ref_err)


def test_many_layouts_in_one_call():
    """One call over 2,500 random layouts: far more new layouts than the context's cache of small device tables holds, so
    the per-point inputs must not depend on it.  Points at the start, middle and end equal their composed runs."""
    from ofdm_b200 import part2
    ctx = _ctx("f32")
    rng = np.random.default_rng(77)
    masks = [np.sort(rng.permutation(NC)[:int(rng.integers(16, 200))]) + 1 for _ in range(2500)]
    kw = dict(profile="EPA", fs_hz=FS, snr_db=SNR, seed=31)
    _, _, per, counts, rn = part2.sweep_lib(ctx, [0] * len(masks), 1, ALL_BITS, reg_pilot=False, random_masks=masks, **kw)
    assert np.all(rn[:, 0] == 1) and np.all(np.isfinite(per)) and np.all(per > 0)
    for k in (0, 1250, 2499):
        pc, dc = part2.layout(NC, pilotCarriers=masks[k])
        nmse, errs, _, _ = part2.run_point(ctx, pc, dc, ALL_BITS[:S * dc.size * 4], 1, point_id=k, first_run=0, Ldict=NFFT, **kw)
        assert np.array_equal(per[k].T, nmse) and np.array_equal(counts[k, :, 0], errs), k


def test_the_experiment_is_sane():
    from ofdm_b200 import part2
    ctx = _ctx("f32")
    NMSE, BER, per, _, _ = part2.sweep_lib(ctx, [8], 16, ALL_BITS, profile="EVA", fs_hz=FS, snr_db=SNR, seed=9)
    assert np.all(np.isfinite(per)) and np.all(per > 0)
    assert BER[0, 0] < 0.05                              # LS with 128 pilots at 20 dB on EVA: a working link
    NMSE, _, _, _, _ = part2.sweep_lib(ctx, [4, 64], 100, ALL_BITS, profile="EPA", fs_hz=FS, snr_db=SNR, seed=3)
    assert NMSE[0, 0] < NMSE[0, 1]                       # denser pilots, better LS estimate


def test_mex_gateway_equals_python():
    import os
    import subprocess
    from ofdm_b200 import part2
    from test_gpu_mex import Mex
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["make", "-C", os.path.join(root, "mex")], check=True, capture_output=True)
    mex = Mex("interleaved")
    ctx = _ctx("f32")
    from ofdm_b200 import link as G
    amp = 2.0 * float(np.max(np.abs(G.constellation_func("16QAM")[0])))
    mask = np.sort(np.random.default_rng(8).permutation(NC)[:64]) + 1
    runs, seed = 5, 4
    bits = ALL_BITS[:S * (NC - 4) * 4]
    kw = dict(profile="ETU", fs_hz=FS, snr_db=SNR, seed=seed, near_eps=1e-3, tie_eps=1e-3)
    scal = [float(NFFT), float(NFFT // 8), float(NC), float(S), 7.0, "16QAM"]
    tail = [part2.pilot_pattern(amp), bits.astype(float), "ETU", FS, SNR, float(runs), float(seed), 1e-3, 1e-3]
    try:
        for pil, off, want in ((np.array([[37.0, 256.0]]), np.zeros(0), part2.sweep_lib(ctx, [37, 256], runs, bits, **kw)),
                               (mask[None].astype(float), np.array([[0.0, 64.0]]),
                                part2.sweep_lib(ctx, [0], runs, bits, reg_pilot=False, random_masks=[mask], **kw))):
            got = mex.call("sweep_part2", *scal, pil, off, np.zeros(0), *tail, nout=5)
            P = want[0].shape[1]
            assert np.allclose(got[0], want[0], rtol=1e-13, atol=0)         # the gateway sums the runs in order
            assert np.array_equal(got[1], want[1])
            assert np.array_equal(got[2].reshape(runs, 4, P, order="F").transpose(2, 1, 0), want[2])
            assert np.array_equal(got[3].reshape(3, 4, P, order="F").transpose(2, 1, 0).astype(np.int64), want[3])
            assert np.array_equal(got[4].T.astype(np.int64), want[4])
    finally:
        mex.lib.ofdm_mex_shim_exit()


def test_rejections():
    from ofdm_b200 import _cabi, part2
    keep = []

    def call(combs=(4, 8), offsets=None, carriers=None, ldict=None, payload_bits=None, base=None, null=None, c=None, **over):
        ctx = c or _ctx("f32")
        off, car, ld = part2.lib_layout(list(combs))
        off = np.ascontiguousarray(off if offsets is None else offsets, dtype=np.int32)
        car = np.ascontiguousarray(car if carriers is None else carriers, dtype=np.int32)
        ld = np.ascontiguousarray(ld if ldict is None else ldict, dtype=np.int32)
        pat = np.ascontiguousarray(part2.pilot_pattern(1.9))
        words = np.zeros(S * NC * 4 // 32, dtype=np.uint32)
        keep.extend([off, car, ld, pat, words])
        lp = _cabi.LinkParams()
        lp.Nfft, lp.Tg, lp.N_carrier, lp.S, lp.SpF, lp.constellation = NFFT, NFFT // 8, NC, S, 7, 4
        for f, v in (base or {}).items():
            setattr(lp, f, v)
        pp = _cabi.Part2Params()
        pp.n_points = ld.size
        pp.pilot_offsets_host, pp.pilot_carriers_host = off.ctypes.data_as(_cabi.pi32), car.ctypes.data_as(_cabi.pi32)
        pp.ldict_host, pp.pilot_pattern_host = ld.ctypes.data_as(_cabi.pi32), pat.ctypes.data_as(_cabi.pdbl)
        pp.payload_host, pp.payload_bits = words.ctypes.data_as(C.POINTER(C.c_uint32)), S * NC * 4 if payload_bits is None else payload_bits
        pp.profile, pp.fs_hz, pp.snr_db, pp.mc_runs, pp.rank, pp.world, pp.seed = 0, FS, SNR, 2, 0, 1, 1
        for f, v in over.items():
            setattr(pp, f, v)
        per = torch.zeros((max(ld.size, 1), 4, 2), dtype=torch.float64, device=ctx.device)
        cnt = torch.zeros((max(ld.size, 1), 4, 3), dtype=torch.int64, device=ctx.device)
        rn = torch.zeros((max(ld.size, 1), 2), dtype=torch.int64, device=ctx.device)
        args = [C.byref(lp), C.byref(pp), ctx.p(per), ctx.p(cnt), ctx.p(rn)]
        if null is not None:
            args[null] = None
        rc = ctx.lib.ofdm_sweep_part2(ctx.h, *args)
        ctx.sync()
        return rc, ctx.lib.ofdm_last_error(ctx.h).decode()

    assert call()[0] == 0
    cases = [
        (dict(null=0), "null pointer"), (dict(null=1), "null pointer"), (dict(null=2), "null pointer"), (dict(null=3), "null pointer"),
        (dict(null=4), "null pointer"),
        (dict(pilot_pattern_host=None), "null host array"),
        (dict(n_points=0), "at least one sweep point"),
        (dict(offsets=[0, 256, 250]), "non-decreasing"),
        (dict(offsets=[1, 256, 384]), "start at 0"),
        (dict(combs=(4, 1025)), "at least two pilots"),
        (dict(carriers=np.r_[np.arange(1, 1025, 4)[::-1], np.arange(1, 1025, 8)]), "strictly increasing"),
        (dict(combs=(1,)), "at least one data carrier"),
        (dict(ldict=[255, 512]), "Np <= Ldict <= Nfft"),
        (dict(ldict=[1024, 4097]), "Np <= Ldict <= Nfft"),
        (dict(profile=2, fs_hz=1e9), "not be longer than N_carrier"),
        (dict(payload_bits=S * 896 * 4 - 1), "payload_bits is shorter"),
        (dict(profile=3), "profile must be"),
        (dict(fs_hz=0.0), "fs_hz must be positive"),
        (dict(mc_runs=0), "mc_runs must be in"),
        (dict(mc_runs=1_000_004), "mc_runs must be in"),
        (dict(tile_runs=-1), "tile_runs must be"),
        (dict(rank=1, world=1), "bad rank / world"),
        (dict(base={"Nfft": 16384, "Tg": 2048}), "Nfft must be a power of two"),
        (dict(base={"Nfft": 3000}), "Nfft must be a power of two"),
    ]
    for kw, text in cases:
        rc, msg = call(**kw)
        assert rc == -1 and text in msg, (kw, rc, msg)
    rc, msg = call(c=_ctx("f64"), base={"Nfft": 8192, "Tg": 1024})
    assert rc == -1 and "8..4096 in FP64" in msg
    # K = n_paths <= 32 cannot fail with the three 3GPP profiles (at most 9 paths); the check guards the pursuit kernels.
