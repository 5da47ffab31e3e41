"""ofdm_group (one host call, several GPUs of the process): every sweep through a group is bit-identical to the single-context
call with world 1 on device 0 -- integers exactly, float cells as their bit patterns (NaN payloads and -0.0 count) -- for
groups with a repeated device, two GPUs and all GPUs; more members than streams; member errors; the caller's current device;
and the MEX gateway's 'devices' op in both complex-storage variants."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as O
from oracle import chains as OC

pytestmark = pytest.mark.gpu

TAPS5 = [[0, 1], [4, .8], [10, .6], [15, .4], [21, .2], [25, .1]]     # `Main_model_Task_5.m:112-119`
TAPS4 = [[0, 1], [4, .6], [10, .3]]                                   # `Task 4/Main_model_Task_4.m:252-264`
NC, S = 1024, 14
PART2_BITS = np.random.default_rng(2024).integers(0, 2, S * NC * 4).astype(np.uint8)
GROUP_SETS = {"repeat0": lambda n: [0, 0], "pair01": lambda n: [0, 1] if n >= 2 else None,
              "all": lambda n: list(range(n)) if n >= 3 else None}
_groups = {}


def _group(devices, prec="f32"):
    import ofdm_b200 as G
    key = (tuple(devices), prec)
    if key not in _groups:
        _groups[key] = G.Group(devices, prec)
    return _groups[key]


@pytest.fixture(scope="module", autouse=True)
def _close_groups():
    yield
    for g in _groups.values():
        g.close()
    _groups.clear()


@pytest.fixture(scope="module", params=list(GROUP_SETS))
def devices(request):
    devs = GROUP_SETS[request.param](torch.cuda.device_count())
    if devs is None:
        pytest.skip(f"{request.param} needs more GPUs than {torch.cuda.device_count()}")
    return devs


def _ctx(prec="f32"):
    import ofdm_b200 as G
    return G.default_context(prec)


def _lp(ctx, p, scramble=True):
    return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                           p.pilotCarriers, p.pilotValues, scramble=scramble)


def _same(got, want):
    """bit-identical: int64 exactly, float64 by bit pattern"""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want.cpu().numpy() if isinstance(want, torch.Tensor) else want)
    assert got.shape == want.shape and got.dtype == want.dtype
    assert np.array_equal(got.view(np.int64), want.view(np.int64))


@pytest.mark.parametrize("chain", ["task5", "task4"])
def test_sweep_ber(devices, chain):
    from ofdm_b200 import sweep
    ctx = _ctx()
    p, taps = (OC.params_task5(comb=4), TAPS5) if chain == "task5" else (OC.params_task4(), TAPS4)
    lp = _lp(ctx, p)
    kw = dict(taps=taps, chain=chain, seed=7, tile=77, near_eps=1e-3)
    want = sweep.sweep_local(ctx, lp, [4.0, 12.0, 20.0], 301, **kw)
    got = _group(devices).sweep_ber(lp, [4.0, 12.0, 20.0], 301, **kw)
    ctx.sync()
    _same(got, want)
    assert np.all(got[:, 1] == 301 * p.stream_bits) and got[0, 0] > got[2, 0]


def test_sweep_mse(devices):
    from ofdm_b200 import sweep
    ctx = _ctx()
    lp = _lp(ctx, OC.params_task5(comb=4))
    kw = dict(seed=5, tile=61, tie_eps=1e-3)
    per, cnt = sweep.mse_sweep_local(ctx, lp, [6.0, 18.0], 257, TAPS5, **kw)
    got_per, got_cnt = _group(devices).sweep_mse(lp, [6.0, 18.0], 257, TAPS5, **kw)
    ctx.sync()
    _same(got_per, per)
    _same(got_cnt, cnt)
    assert np.all(got_cnt[:, 0] == 257)


@pytest.mark.parametrize("fixed", [False, True])
def test_sweep_sync(devices, fixed):
    from ofdm_b200 import sweep
    ctx = _ctx()
    lp = _lp(ctx, OC.params_task4())
    kw = dict(seed=3, tile=97, sto=150, cfo=0.24, mp_desync=False) if fixed else dict(seed=3, tile=97)
    rec, cnt = sweep.sync_sweep_local(ctx, lp, [0.0, 15.0], 263, TAPS4, **kw)
    got_rec, got_cnt = _group(devices).sweep_sync(lp, [0.0, 15.0], 263, TAPS4, **kw)
    ctx.sync()
    _same(got_rec, rec)
    _same(got_cnt, cnt)


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_sweep_papr(devices, prec):
    from ofdm_b200 import sweep
    ctx = _ctx(prec)
    lp = _lp(ctx, OC.params_task4(percent=1, scale=2.0, alternate=True))
    pts = [(0, 0.5), (1, 0.5), (0, 0.05)]
    kw = dict(seed=9, tile=71, bin_db=0.05, n_bins=300)
    hist, papr = sweep.papr_sweep_local(ctx, lp, pts, 211, **kw)
    got_hist, got_papr = _group(devices, prec).sweep_papr(lp, pts, 211, **kw)
    ctx.sync()
    _same(got_hist, hist)
    _same(got_papr, papr)


def test_sweep_part2(devices):
    from ofdm_b200 import part2
    ctx = _ctx()
    kw = dict(profile="ETU", fs_hz=4e7, snr_db=20.0, seed=4, near_eps=1e-3, tie_eps=1e-3)
    per, cnt, runs = part2.sweep_lib_local(ctx, [4, 37, 256], 53, PART2_BITS, tile=9, **kw)
    got = _group(devices).sweep_part2([4, 37, 256], 53, PART2_BITS, tile=9, **kw)
    ctx.sync()
    for g, w in zip(got, (per, cnt, runs)):
        _same(g, w)
    assert np.all(got[2][:, 0] == 53)


def test_more_members_than_streams():
    from ofdm_b200 import sweep
    ctx = _ctx()
    p = OC.params_task5(comb=4)
    lp = _lp(ctx, p)
    want = sweep.sweep_local(ctx, lp, [10.0], 2, TAPS5, seed=2)
    got = _group([0, 0, 0]).sweep_ber(lp, [10.0], 2, TAPS5, seed=2)
    ctx.sync()
    _same(got, want)
    assert got[0, 1] == 2 * p.stream_bits


def test_member_errors_and_recovery():
    import ofdm_b200 as G
    from ofdm_b200 import sweep
    ctx = _ctx()
    lp = _lp(ctx, OC.params_task5(comb=4))
    g = _group([0, 0])
    with pytest.raises(G.OfdmError) as single:
        sweep.sweep_local(ctx, lp, [], 10, TAPS5)
    with pytest.raises(G.OfdmError, match=r"device 0 \(member 0\): .*SNR point") as grp:
        g.sweep_ber(lp, [], 10, TAPS5)
    assert grp.value.status == -1 and str(single.value).startswith("status -1:")
    # FP64 contexts do not run the sync sweep: the single call's status, then the same group runs a valid call
    ctx64 = _ctx("f64")
    lp4 = _lp(ctx64, OC.params_task4())
    with pytest.raises(G.OfdmError, match="status -4"):
        sweep.sync_sweep_local(ctx64, lp4, [10.0], 5, TAPS4)
    g64 = _group([0, 0], "f64")
    with pytest.raises(G.OfdmError, match=r"member 0\): ofdm_sweep_sync runs the FP32") as e:
        g64.sweep_sync(lp4, [10.0], 5, TAPS4)
    assert e.value.status == -4
    lp5 = _lp(ctx64, OC.params_task5(comb=4))
    want = sweep.sweep_local(ctx64, lp5, [8.0, 16.0], 40, TAPS5, seed=6, tile=13)
    _same(g64.sweep_ber(lp5, [8.0, 16.0], 40, TAPS5, seed=6, tile=13), want)


def test_create_rejections():
    from ofdm_b200 import _cabi
    lib = _cabi.load()
    n = torch.cuda.device_count()
    for ids, count, status in (([0], 0, -1), (None, 2, -1), ([0, n], 2, -3), ([-1], 1, -3)):
        h = C.c_void_p(1)
        arr = None if ids is None else (C.c_int32 * len(ids))(*ids)
        assert lib.ofdm_group_create(C.byref(h), arr, count, 0) == status
        assert not h.value
    lib.ofdm_group_destroy(None)
    g = _group([0, 0])
    assert lib.ofdm_group_size(g.h) == 2


def test_current_device_is_preserved():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from ofdm_b200 import _cabi, sweep
    lib = _cabi.load()
    ctx = _ctx()
    lp = _lp(ctx, OC.params_task5(comb=4))
    before_dev = torch.cuda.current_device()
    before = sweep.ber_sweep(ctx, lp, [9.0], 64, TAPS5, seed=11)
    h = C.c_void_p()
    ids = (C.c_int32 * 2)(0, 1)
    assert lib.ofdm_group_create(C.byref(h), ids, 2, 0) == 0
    try:
        assert torch.cuda.current_device() == before_dev
        torch.zeros(4, device="cuda").add_(1)
        assert np.array_equal(sweep.ber_sweep(ctx, lp, [9.0], 64, TAPS5, seed=11), before)
    finally:
        lib.ofdm_group_destroy(h)
    assert torch.cuda.current_device() == before_dev


# ---------------------------------------------------------------- MEX gateway
def _link_args(p):
    return [float(p.Nfft), float(p.T_Guard), float(p.N_carrier), float(p.N_symb), float(p.Amount_ODFM_SpF), p.Constellation,
            p.dataCarriers.astype(float), p.pilotCarriers.astype(float), p.pilotValues, O.DEFAULT_REGISTER.astype(float)]


@pytest.fixture(scope="module", params=["interleaved", "split"])
def mex(request):
    import os
    import subprocess
    from test_gpu_mex import Mex
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["make", "-C", os.path.join(root, "mex")], check=True, capture_output=True)
    m = Mex(request.param)
    yield m
    m.call("devices", 0.0)
    m.lib.ofdm_mex_shim_exit()


def _mex_sweeps(mex):
    """every sweep op once, at shapes the shim converts quickly"""
    p5, p4, p2 = OC.params_task5(comb=4), OC.params_task4(), OC.params_task4(percent=1, scale=2.0, alternate=True)
    amp = 2.0 * float(np.max(np.abs(O.constellation_func("16QAM")[0])))
    from ofdm_b200 import part2
    out = [mex.call("sweep_ber", *_link_args(p5), np.array([5.0, 15.0]), 7.0, np.asarray(TAPS5, dtype=float), "task5", 3.0, 1e-3),
           mex.call("sweep_ber", *_link_args(p4), np.array([10.0, 30.0]), 5.0, np.asarray(TAPS4, dtype=float), "task4", 3.0, 1e-3)]
    out += mex.call("sweep_mse", *_link_args(p5), np.array([5.0, 15.0]), 5.0, np.asarray(TAPS5, dtype=float), 3.0, 1e-3, nout=3)
    out += mex.call("sweep_sync", *_link_args(p4), np.array([5.0, 15.0]), 7.0, np.asarray(TAPS4, dtype=float), 3.0, -1.0, 0.0,
                    np.array([1.0, 1.0, 1.0]), nout=2)
    out += mex.call("sweep_papr", *_link_args(p2), np.array([0.0, 1.0]), np.array([0.5, 0.5]), 5.0, 3.0, 0.05, 200.0, np.zeros((0, 0)),
                    0.0, nout=2)
    out += mex.call("sweep_part2", float(4096), float(512), float(NC), float(S), 7.0, "16QAM", np.array([[37.0, 256.0]]), np.zeros(0),
                    np.zeros(0), part2.pilot_pattern(amp), PART2_BITS[:S * (NC - 4) * 4].astype(float), "ETU", 4e7, 20.0, 5.0, 4.0,
                    1e-3, 1e-3, nout=5)
    return out


def test_mex_devices(mex):
    assert np.array_equal(mex.call("devices"), [[0.0]])
    want = _mex_sweeps(mex)
    try:
        assert np.array_equal(mex.call("devices", np.array([0.0, 0.0])), [[0.0, 0.0]])
        assert np.array_equal(mex.call("devices"), [[0.0, 0.0]])
        got = _mex_sweeps(mex)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert g.shape == w.shape and np.array_equal(np.ascontiguousarray(g).view(np.int64), np.ascontiguousarray(w).view(np.int64))
        with pytest.raises(RuntimeError, match="ofdm:devices:id"):
            mex.call("devices", np.array([0.0, -1.0]))
        with pytest.raises(RuntimeError, match="ofdm:devices:nodevice"):
            mex.call("devices", float(torch.cuda.device_count()))
        assert np.array_equal(mex.call("devices"), [[0.0]])                  # a set that failed to build falls back to [0]
    finally:
        mex.call("devices", 0.0)
