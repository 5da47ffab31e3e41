"""ofdm_sweep_papr (csrc/sweep_papr.cu + papr_stats_kernel in csrc/papr.cu): the Task-2 PAPR study as one library call per
rank.  The histogram must equal, bin for bin, the composed exported calls payload -> ofdm_tx_chain -> ofdm_window_papr -> the
bin rule on the host; the per-stream PAPR must agree with ofdm_papr; and the results must not depend on the tile size or the
rank count.  P4 and P7 (`Task 2/README.md:54,69-71`) are checked through the call on the eagle payload."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import oracle as O
from oracle import chains as OC

import reference_pins as RP

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P7 = {"plain": 21.878, "scrambled": 10.911}          # oracle regression values, as in tests/test_papr_pins.py
STRIDE = 1237


@pytest.fixture(scope="module")
def G():
    import ofdm_b200
    return ofdm_b200


def _ctx(prec="f32"):
    import ofdm_b200
    return ofdm_b200.default_context(prec)


def _lp(ctx, p, scramble=True):
    return ctx.link_params(p.Nfft, p.T_Guard, p.N_carrier, p.N_symb, p.Amount_ODFM_SpF, p.Constellation, p.dataCarriers,
                           p.pilotCarriers, p.pilotValues, scramble=scramble)


LAYOUTS = {"task2": lambda: OC.params_task4(percent=1, scale=2.0, alternate=True),    # Nfft 1024, 79,000-bit streams, tx1024
           "task5": lambda: OC.params_task5(comb=4)}                                  # Nfft 4096, tx4096


def _pool_payload(pool, n, stream_bits, stride, first=0):
    j = np.arange(first, first + n, dtype=np.int64)[:, None]
    i = np.arange(stream_bits, dtype=np.int64)[None, :]
    return pool[(j * stride + i) % pool.size]


def _composed(ctx, p, scramble, bits_dev, n, bin_db, n_bins):
    """payload -> ofdm_tx_chain -> ofdm_window_papr -> host bin rule; and ofdm_papr.  Returns (hist, papr)."""
    tx = ctx.tx_chain(_lp(ctx, p, bool(scramble)), bits_dev, n).reshape(n, -1)
    w = ctx.window_papr(tx, p.Nfft).cpu().numpy().astype(np.float64)
    q = np.floor(w / bin_db)
    b = np.where(q > 0, np.minimum(q, n_bins - 1), 0).astype(np.int64)
    return np.bincount(b.ravel(), minlength=n_bins), ctx.papr(tx).cpu().numpy()


@pytest.mark.parametrize("prec", ["f32", "f64"])
@pytest.mark.parametrize("layout", ["task2", "task5"])
@pytest.mark.parametrize("payload", ["bernoulli", "pool"])
def test_bit_identity_with_composed_calls(G, prec, layout, payload):
    from ofdm_b200 import sweep
    ctx = _ctx(prec)
    p = LAYOUTS[layout]()
    spp, bin_db, n_bins = 3, 0.01, 3000
    tol = 1e-10 if prec == "f64" else 1e-4
    pool = RP.eagle_bits(200000) if payload == "pool" else None
    pone = 0.05
    hist, papr = sweep.papr_sweep_local(ctx, _lp(ctx, p), [(0, pone), (1, pone)], spp, seed=5, bin_db=bin_db, n_bins=n_bins, pool=pool,
                                        pool_stride=STRIDE)
    ctx.sync()
    hist, papr = hist.cpu().numpy(), papr.cpu().numpy()
    if pool is None:
        bits_dev = ctx.payload_bernoulli(spp, p.stream_bits, pone, seed=5)
    else:
        bits_dev = ctx.bits(_pool_payload(pool, spp, p.stream_bits, STRIDE).ravel())
    L = p.N_symb * (p.Nfft + p.T_Guard)
    for k, scr in enumerate((0, 1)):
        h_ref, p_ref = _composed(ctx, p, scr, bits_dev, spp, bin_db, n_bins)
        assert np.array_equal(hist[k], h_ref), (k, np.flatnonzero(hist[k] != h_ref)[:10])
        assert hist[k].sum() == spp * (L - p.Nfft + 1)
        assert np.max(np.abs(papr[k] - p_ref)) <= tol
    if pool is None:
        assert np.all(papr[0] > papr[1])             # the scrambler flattens a biased payload


def test_tile_and_rank_invariance(G):
    from ofdm_b200 import sweep
    ctx = _ctx("f32")
    p = LAYOUTS["task2"]()
    lp = _lp(ctx, p)
    pts, spp = [(0, 0.3), (1, 0.3)], 800
    kw = dict(seed=9, bin_db=0.02, n_bins=1500)
    ref_h, ref_p = sweep.papr_sweep_local(ctx, lp, pts, spp, **kw)
    L = p.N_symb * (p.Nfft + p.T_Guard)
    for tile in (1, 777):
        h, pa = sweep.papr_sweep_local(ctx, lp, pts, spp, tile=tile, **kw)
        assert torch.equal(h, ref_h) and torch.equal(pa, ref_p), tile
    h = torch.zeros_like(ref_h)
    pa = torch.zeros_like(ref_p)
    for r in range(3):
        sweep.papr_sweep_local(ctx, lp, pts, spp, rank=r, world=3, tile=300, hist=h, papr=pa, **kw)
    assert torch.equal(h, ref_h) and torch.equal(pa, ref_p)
    assert np.all(ref_h.sum(dim=1).cpu().numpy() == spp * (L - p.Nfft + 1))


@pytest.mark.parametrize("prec,ptol", [("f64", 1e-6), ("f32", 1e-4)])
def test_P4_P7_through_the_call(G, prec, ptol):
    """The eagle payload as the pool, one stream per point, stride 0: the reference's own experiment."""
    from ofdm_b200 import sweep
    ctx = _ctx(prec)
    p = LAYOUTS["task2"]()
    bits = RP.eagle_bits(p.stream_bits)
    # 16,384 bins of 0.001 dB end at 16.4 dB, below the plain figure: the finest histogram reaching 22 dB has 0.002 dB bins
    bin_db, n_bins = 0.002, 16384
    res = sweep.papr_sweep(ctx, _lp(ctx, p), [(0, None), (1, None)], 1, bin_db=bin_db, n_bins=n_bins, pool=bits, pool_stride=0)
    ex = sweep.papr_exceedance(res["hist"], bin_db, 0.02)
    for k, scr in enumerate((False, True)):
        tx = OC.tx_chain(p, bits, scramble=scr, fast=True)[0]
        assert abs(res["papr"][k, 0] - O.calculatePAPR(tx)) < ptol
        x, c = O.calculateCCDF(O.calculate_window_PAPR(tx, p.Nfft))
        v = x[np.argmax(c <= 0.02)]
        assert abs(v - P7["scrambled" if scr else "plain"]) < 0.01
        assert abs(ex[k] - v) <= bin_db + 1e-3, (k, ex[k], v)
        assert abs(res["papr"][k, 0] - RP.PAPR_T2["scrambled" if scr else "plain"]) < 1.5      # P4
        assert abs(ex[k] - RP.PAPR_T2["scrambled" if scr else "plain"]) < 1.5                   # P7 against the README's 22 / 10


def test_scrambler_study_statistics(G):
    """A biased payload makes the plain signal peaky and the scrambler removes it; an unbiased one is already noise-like."""
    from ofdm_b200 import sweep
    ctx = _ctx("f32")
    p = LAYOUTS["task2"]()
    res = sweep.papr_sweep(ctx, _lp(ctx, p), [(0, 0.05), (1, 0.05), (0, 0.5), (1, 0.5)], 64, seed=2)
    ex = sweep.papr_exceedance(res["hist"], 0.01, 0.02)
    assert ex[0] - ex[1] > 8.0, ex
    assert abs(ex[2] - ex[3]) < 0.5, ex


def _philox(c, key):
    """Philox4x32-10 on uint32 arrays c (4, n) (csrc/philox.cuh)."""
    c = [x.astype(np.uint64) for x in c]
    k0, k1 = np.uint64(key & 0xFFFFFFFF), np.uint64(key >> 32)
    m = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return c


def test_payload_bernoulli(G):
    from ofdm_b200 import link
    ctx = _ctx("f32")
    sb = 79000
    whole = ctx.payload_bernoulli(10, sb, 0.05, seed=4)
    parts = [ctx.payload_bernoulli(4, sb, 0.05, seed=4), ctx.payload_bernoulli(6, sb, 0.05, seed=4, first_stream_id=4)]
    ctx.sync()
    a = link.unpack_bits(whole.cpu().numpy().view(np.uint32), 10 * sb)
    b = np.concatenate([link.unpack_bits(t.cpu().numpy().view(np.uint32), n * sb) for t, n in zip(parts, (4, 6))])
    assert np.array_equal(a, b)
    # the rule, on the host: bit i of stream j is 1 iff word i mod 4 of Philox at (i / 4, j) < floor(p 2^32)
    j, i = 7, np.arange(4000)
    q = i // 4
    c = _philox([q.astype(np.uint32), np.zeros_like(q, dtype=np.uint32), np.full(q.size, j, np.uint32), np.zeros(q.size, np.uint32)],
                4 ^ 0x6265726e6f756c6c)
    u = np.stack(c)[i % 4, np.arange(i.size)]
    assert np.array_equal(a.reshape(10, sb)[j, :4000], (u < np.uint64(int(0.05 * 2 ** 32))).astype(np.uint8))
    for pone in (0.05, 0.5):
        n = 127                                            # 10.03 M bits
        w = ctx.payload_bernoulli(n, sb, pone, seed=11)
        ones = int(np.unpackbits(w.cpu().numpy().view(np.uint8)).sum())
        N = n * sb
        assert abs(ones / N - pone) < 5 * np.sqrt(pone * (1 - pone) / N)
    t = ctx.payload_bernoulli(3, sb, 0.9, seed=1).cpu().numpy().view(np.uint32)
    assert t.size == (3 * sb + 31) // 32 and (int(t[-1]) >> ((3 * sb) % 32)) == 0     # bits past the last stream are 0


def test_arguments(G):
    from ofdm_b200 import _cabi
    ctx = _ctx("f32")
    p = LAYOUTS["task2"]()
    lp = _lp(ctx, p)
    hist = torch.zeros((2, 100), dtype=torch.int64, device=ctx.device)
    papr = torch.zeros((2, 4), dtype=torch.float64, device=ctx.device)
    scr = np.array([0, 1], dtype=np.int32)
    bad_scr = np.array([0, 2], dtype=np.int32)
    pone = np.array([0.5, 0.5])
    bad_pone = np.array([0.5, 1.0])
    pool = np.ones(4, dtype=np.uint32)

    def params(**kw):
        pp = _cabi.PaprParams()
        pp.n_points, pp.streams_per_point, pp.rank, pp.world, pp.seed, pp.bin_db, pp.n_bins = 2, 4, 0, 1, 1, 0.1, 100
        pp.scramble_host = scr.ctypes.data_as(_cabi.pi32)
        pp.p_one_host = pone.ctypes.data_as(_cabi.pdbl)
        for k, v in kw.items():
            setattr(pp, k, v)
        return pp

    def call(pp, l=lp, c=ctx, pa=papr, hi=hist):
        rc = c.lib.ofdm_sweep_papr(c.h, C.byref(l) if l is not None else None, C.byref(pp) if pp is not None else None, c.p(pa), c.p(hi))
        return rc, c.lib.ofdm_last_error(c.h).decode()

    assert call(params())[0] == 0
    cases = [
        (dict(l=None), "link parameters"), (dict(pp=None), "PAPR parameters"), (dict(pa=None), "papr_dev"), (dict(hi=None), "hist_dev"),
        (dict(n_points=0), "point"), (dict(scramble_host=None), "scramble_host"),
        (dict(scramble_host=bad_scr.ctypes.data_as(_cabi.pi32)), "scramble flags"), (dict(p_one_host=None), "p_one_host"),
        (dict(p_one_host=bad_pone.ctypes.data_as(_cabi.pdbl)), "p_one"),
        (dict(pool_host=pool.ctypes.data_as(C.POINTER(C.c_uint32)), pool_bits=0), "pool_bits"),
        (dict(pool_host=pool.ctypes.data_as(C.POINTER(C.c_uint32)), pool_bits=100, pool_stride=-1), "pool_stride"),
        (dict(streams_per_point=0), "stream per point"), (dict(tile_streams=-1), "tile_streams"), (dict(rank=1, world=1), "rank"),
        (dict(world=0), "rank"), (dict(bin_db=0.0), "bin_db"), (dict(bin_db=float("inf")), "bin_db"), (dict(n_bins=0), "n_bins"),
        (dict(n_bins=16385), "n_bins"),
    ]
    texts = set()
    for kw, needle in cases:
        call_kw = {k: kw.pop(k) for k in ("l", "pa", "hi") if k in kw}
        pp = None if kw.pop("pp", 0) is None else params(**kw)
        rc, text = call(pp, **call_kw)
        assert rc == -1 and needle in text, (kw, call_kw, rc, text)
        texts.add(text)
    assert len(texts) == len(cases) - 3                     # the two rank, bin_db and n_bins cases share their texts
    # the statistics kernel's shared memory: FP32 at Nfft 8192 with 16,384 bins needs 256 KB per block
    l8 = ctx.link_params(8192, 0, 400, 5, 5, "QPSK", np.arange(3, 401), [1, 2], np.ones((2, 5)))
    h8 = torch.zeros((2, 16384), dtype=torch.int64, device=ctx.device)
    rc, text = call(params(n_bins=16384), l=l8, hi=h8)
    assert rc == -4 and "shared memory" in text and "Nfft 8192" in text
    assert call(params(n_bins=4000), l=l8, hi=h8)[0] == 0
    w = torch.zeros(10, dtype=torch.int32, device=ctx.device)
    for args, needle in (((w, 1, 0, 0.5, 1, 0), "stream_bits"), ((w, -1, 8, 0.5, 1, 0), "n_streams"), ((w, 1, 8, 0.0, 1, 0), "p_one"),
                         ((w, 1, 8, 1.0, 1, 0), "p_one"), ((w, 1, 8, 0.5, 1, -1), "first_stream_id"), ((None, 1, 8, 0.5, 1, 0), "bits_dev")):
        rc = ctx.lib.ofdm_payload_bernoulli(ctx.h, ctx.p(args[0]), *args[1:])
        assert rc == -1 and needle in ctx.lib.ofdm_last_error(ctx.h).decode(), args


@pytest.fixture(scope="module")
def mex():
    from test_gpu_mex import Mex
    subprocess.run(["make", "-C", os.path.join(ROOT, "mex")], check=True, capture_output=True)
    m = Mex("interleaved")
    yield m
    m.lib.ofdm_mex_shim_exit()


def test_mex_sweep_papr_equals_python(G, mex):
    from ofdm_b200 import sweep
    ctx = _ctx("f32")
    p = LAYOUTS["task2"]()
    lp = _lp(ctx, p)
    reg = O.DEFAULT_REGISTER.astype(float)
    args = [float(p.Nfft), float(p.T_Guard), float(p.N_carrier), float(p.N_symb), float(p.Amount_ODFM_SpF), p.Constellation,
            p.dataCarriers.astype(float), p.pilotCarriers.astype(float), p.pilotValues, reg]
    spp, bin_db, n_bins = 5, 0.05, 600
    got_h, got_p = mex.call("sweep_papr", *args, np.array([0.0, 1.0]), np.array([0.05, 0.05]), float(spp), 3.0, bin_db, float(n_bins),
                            np.zeros((0, 0)), 0.0, nout=2)
    res = sweep.papr_sweep(ctx, lp, [(0, 0.05), (1, 0.05)], spp, seed=3, bin_db=bin_db, n_bins=n_bins)
    assert got_h.shape == (n_bins, 2) and got_p.shape == (spp, 2)
    assert np.array_equal(got_h.T.astype(np.int64), res["hist"])
    assert np.array_equal(got_p.T, res["papr"])
    pool = RP.eagle_bits(p.stream_bits)
    got_h, got_p = mex.call("sweep_papr", *args, np.array([0.0, 1.0]), np.array([0.5, 0.5]), 2.0, 1.0, bin_db, float(n_bins),
                            pool.astype(float), 17.0, nout=2)
    res = sweep.papr_sweep(ctx, lp, [(0, None), (1, None)], 2, bin_db=bin_db, n_bins=n_bins, pool=pool, pool_stride=17)
    assert np.array_equal(got_h.T.astype(np.int64), res["hist"]) and np.array_equal(got_p.T, res["papr"])
